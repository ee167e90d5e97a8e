// pcm1_kernels.cuh -- PCM-1 line decode kernels (device only).
//
//   pcm1_prescan_kernel : VideoToDigital::prescanCoordinates for every frame at once -- four full coordinate searches
//                         per frame (Binarizer reset, so a pure function of the frame), one thread block per search,
//                         one grid point per thread.
//   pcm1_preset_kernel  : median of the four results -> per-frame presets (reference level, data coordinates).
//   pcm1_bulk_kernel    : the HBM-bound pass.  One warp per frame, one lane per video line, 32 rows per step through a
//                         per-warp staging ring of bulk_ring.cuh, as in stc007_bulk_kernel.  Decodes
//                         every line with the frame's presets (STG_INPUT_ALL -> first readPCMdata candidate), finds the
//                         frame's black/white levels from the first non-header line the way the reference's first line
//                         of the frame does, applies the per-field rules of a valid line and flags the frame clean.
//   pcm1_chain_kernel   : one block walks the frames in order.  Runs of clean frames whose coordinates stay within the
//                         damper's limit of their predecessor are skipped in one step; every other frame is decoded
//                         with the exact sequential semantics (pcm1_line.cuh, pcm1_chain.cuh): the bulk pass's records
//                         are hints (re-made in the kernel when the chain holds other presets), hinted lines in the
//                         chain's steady state are finished one per thread, lines without a valid hint get the whole block.
#pragma once
#include "bulk_ring.cuh"
#include "pcm1_chain.cuh"
#include "stc007_bulk.cuh"

namespace sdv {

enum { P1L_THREADS = 256, P1C_CHUNK = 256 };     // chain kernel: records staged per chunk
enum { P1S_THREADS = 128 };                      // prescan kernels: a search is a chain of short phases, few of them wider than 64 threads -- what
                                                 // counts is how many searches an SM holds at once (8 blocks of 128 threads at 64 registers)

// opens: frame 0 of the call opens the file (carries the NEW_FILE line); 0 when the call continues the previous call's file.
__global__ void __launch_bounds__(P1S_THREADS, 8) pcm1_prescan_kernel(const u8 *luma, int H, int W, size_t stride, int n_frames, int mode, int opens, P1Preset *scan)
{
    __shared__ P1Work w;
    __shared__ __align__(16) u8 px[SDV_MAX_W];
    const int f = blockIdx.x/P1_COORD_CHECK_LINES, idx = blockIdx.x%P1_COORD_CHECK_LINES;
    if(f>=n_frames) return;
    P1Preset r; r.valid = 0; r.ref = 0; r.coords = coord_none(); r.pad[0] = r.pad[1] = 0;
    const int row = p1_prescan_row(H, opens&&(f==0), idx);
    if(row<0) { if(threadIdx.x==0) scan[blockIdx.x] = r; return; }
    const u8 *src = luma+((size_t)f*H+(size_t)row)*stride;
    for(int i=threadIdx.x;i<W;i+=blockDim.x) px[i] = __ldg(src+i);
    __syncthreads();
    Cta c = { (int)threadIdx.x, (int)blockDim.x };
    Geom g = make_geom(W);
    BinState b;
    bin_set_mode(&b, mode);
    b.def_coord = coord_none();
    bin_reset_good(&b);
    p1_process_line_cta(c, &w, &b, true, px, g);
    if(threadIdx.x==0)
    {
        if(p1_crc_ok(&w.o)) { r.valid = 1; r.coords = w.o.coords; r.ref = w.o.ref; }
        scan[blockIdx.x] = r;
    }
}

__global__ void pcm1_preset_kernel(const P1Preset *scan, int n_frames, int H, int mode, int opens, P1Preset *presets)
{
    const int f = blockIdx.x*blockDim.x+threadIdx.x;
    if(f>=n_frames) return;
    P1Preset ps; ps.valid = 0; ps.ref = 0; ps.coords = coord_none(); ps.pad[0] = ps.pad[1] = 0;
    if(p1_prescan_runs(H, opens&&(f==0), mode)) ps = p1_prescan_reduce(scan+(size_t)f*P1_COORD_CHECK_LINES);
    presets[f] = ps;
}

struct P1BulkParams                 // pcm1_bulk_kernel and pcm16x0_bulk_kernel
{
    const u8 *luma; int H, W; size_t stride;
    int n_frames;
    const P1Preset *presets;
    const P1Preset *run_g;          // PCM-16x0: presets of the file's first frame (the running pair G), presets[0] or the chain's copy
    int line_dup, mode;
    sdv_line_rec *recs; sdv_line_aux *aux;     // PCM-16x0: three sub-line records per line
    u8 *clean;                      // [n_frames]: 1 = every line of the frame was taken by the kernel
    u32 *frame_bw;                  // [n_frames]: black | white<<8 the frame's (PCM-16x0: last) lines were given
    int use_tma, warps; u32 slot_bytes;
};

enum { P1_BULK_HEADER = BULK_BAR_BYTES+512+BULK_MAX_WARPS*1024 };     // barriers, CRC byte table, one histogram per warp

// Black/white levels of one staged row (findPCM1BW + findBlackWhite tail), by one warp.
__device__ __forceinline__ u32 p1_warp_black_white(const u8 *row, int W, u32 *hist, int lane)
{
    for(int i=lane;i<256;i+=32) hist[i] = 0;
    __syncwarp();
    const int scan_end = W-1;
    const int from = scan_end/8, to = scan_end-scan_end/32;
    for(int i=from+lane;i<to;i+=32) atomicAdd(&hist[row[i]], 1u);
    __syncwarp();
    u32 res = 0;
    if(lane==0)
    {
        u8 bl, wh, st;
        bw_pick_levels(hist, false, &bl, &wh, &st);
        res = (u32)bl|((u32)wh<<8)|((u32)st<<16);
    }
    return __shfl_sync(0xFFFFFFFFu, res, 0);
}

__global__ void __launch_bounds__(BULK_MAX_WARPS*32, 1) pcm1_bulk_kernel(const __grid_constant__ P1BulkParams p)
{
    extern __shared__ __align__(128) u8 dsm[];
    u16 *crc_tab = (u16 *)(dsm+BULK_BAR_BYTES);                 // CRC-16 CCITT byte table
    const int warp = threadIdx.x>>5, lane = threadIdx.x&31;
    u32 *hist = (u32 *)(dsm+BULK_BAR_BYTES+512)+warp*256;
    for(int i=threadIdx.x;i<256;i+=blockDim.x) crc_tab[i] = c_crc8[i];
    BulkRing rb(dsm, P1_BULK_HEADER, p.luma, p.H, p.W, p.stride, 0, p.n_frames, p.use_tma, p.warps, p.slot_bytes);
    __syncthreads();
    rb.prime();

    const int hf = p.H/2;
    const int fld = lane&1;
    const int pixel_stop = p.W-1;

    u32 c01 = 0, c23 = 0, c45 = 0;              // words of this field's last line in the previous step (duplicate check)
    bool c_hdr = false;
    bool frame_bad = false, preset_bad = false;
    // per-frame plan
    int ref = 128; u32 psm = INT_CALC_MULT, half = INT_CALC_MULT/2; int ofs = 0;
    u32 rec5 = 0, rec6 = 0, picked = 0;

    for(long long it=0;it<rb.n_items;it++)
    {
        const BulkItem t = rb.item(it);
        const int f = t.f, b = t.b, r0 = t.r0, rows = t.rows;
        const int k = (r0>>1)+(lane>>1);
        const bool active = lane<rows;
        if(b==0)
        {   // frame presets from the prescan
            const P1Preset ps = p.presets[f];
            Coord cc = ps.coords;
            frame_bad = !(ps.valid&&coord_valid(cc));
            preset_bad = frame_bad;
            if(frame_bad) { cc.start = 0; cc.stop = (i16)(p.W-1); }
            ref = frame_bad ? 128 : ps.ref;
            const Ppb pp = p1_make_ppb(cc);
            psm = pp.psm; half = pp.half; ofs = pp.ofs;
            rec6 = (u32)(u16)cc.start|((u32)(u16)cc.stop<<16);
            // bit cells cut off by the line edges (the forced bit picker only counts them on a valid line)
            P1Line t; t.ppb = pp; t.forced_bad = 0; t.calc_crc = 0; for(int i=0;i<P1L_WORDS;i++) t.words[i] = 0;
            p1_pick_cut_bits(&t, p.mode, pixel_stop, p.W-1);
            picked = (u32)t.picked_left|((u32)t.picked_right<<4);
            c01 = c23 = c45 = 0; c_hdr = false;
        }
        const u8 *stage = rb.acquire(t);
        const u8 *row = stage+(size_t)lane*p.slot_bytes;
        // ---- 94 bit cells of this lane's row
        u32 g[4], ge[4];
        g[3] = 0; ge[3] = 0;
#pragma unroll
        for(int w=0;w<3;w++)
        {
            u32 a = 0, c = 0;
#pragma unroll
            for(int j=0;j<32;j++)
            {
                const int bit = 32*w+j;
                if(bit<P1_BITS)
                {
                    int pos = (int)(((u32)bit*psm+half)>>7)+ofs;
                    pos = max(0, min(pos, pixel_stop-1));
                    const int v = row[pos];
                    a = __funnelshift_l((u32)(ref-v), a, 1);
                    c = __funnelshift_l((u32)(ref-1-v), c, 1);
                }
                else { a <<= 1; c <<= 1; }
            }
            g[w] = a; ge[w] = c;
        }
        const bool any_eq = ((ge[0]^g[0])|(ge[1]^g[1])|(ge[2]^g[2]))!=0;
        if(__any_sync(0xFFFFFFFFu, any_eq)) resolve_equal_cells(g, ge);
        // ---- words and CRCC: CRC over the inverted data bits, result inverted (pcm1line.cpp:158-166)
        const u32 w0 = stream_field<0, 13>(g[0], g[1], g[2], g[3]), w1 = stream_field<13, 13>(g[0], g[1], g[2], g[3]);
        const u32 w2 = stream_field<26, 13>(g[0], g[1], g[2], g[3]), w3 = stream_field<39, 13>(g[0], g[1], g[2], g[3]);
        const u32 w4 = stream_field<52, 13>(g[0], g[1], g[2], g[3]), w5 = stream_field<65, 13>(g[0], g[1], g[2], g[3]);
        const u32 w6 = stream_field<78, 16>(g[0], g[1], g[2], g[3]);
        u32 crc = 0xFFFFu;
        {
            const u32 i0 = ~g[0], i1 = ~g[1], i2 = ~g[2];
            crc = crc16_update((u16)crc, (u16)(i0>>26), 6);                             // bits 0..5
#define P1_MSG_BYTE(J) (stream_field<6+8*(J), 8>(i0, i1, i2, 0u))
#define P1_CRC_STEP(J) crc = ((crc<<8)^crc_tab[((crc>>8)^P1_MSG_BYTE(J))&0xFFu])&0xFFFFu
            P1_CRC_STEP(0); P1_CRC_STEP(1); P1_CRC_STEP(2); P1_CRC_STEP(3); P1_CRC_STEP(4);
            P1_CRC_STEP(5); P1_CRC_STEP(6); P1_CRC_STEP(7); P1_CRC_STEP(8);
#undef P1_CRC_STEP
#undef P1_MSG_BYTE
            crc = (~crc)&0xFFFFu;
        }
        const u32 w01 = w0|(w1<<16), w23 = w2|(w3<<16), w45 = w4|(w5<<16);
        const bool is_hdr = (w01==0x0CCC0666u)&&(w23==0x13331999u)&&(w45==0x0CCC0666u)&&(w6==0xCCCCu);
        const bool crc_ok = (crc==w6)||is_hdr;
        // ---- black/white levels of the frame: what the first non-header line of the frame finds for itself
        if(b==0)
        {
            const bool hdr0 = __shfl_sync(0xFFFFFFFFu, is_hdr ? 1 : 0, 0)!=0;
            u32 bw = p1_warp_black_white(stage+(size_t)(hdr0 ? 2 : 0)*p.slot_bytes, p.W, hist, lane);
            bool ok = ((bw>>16)&1u)&&(ref<(int)((bw>>8)&0xFFu))&&(ref>(int)(bw&0xFFu));
            if(hdr0)
            {   // the header line itself was decoded with its own levels
                const u32 bwh = p1_warp_black_white(stage, p.W, hist, lane);
                ok = ok&&((bwh>>16)&1u)&&(ref<(int)((bwh>>8)&0xFFu))&&(ref>(int)(bwh&0xFFu));
            }
            if(!ok) frame_bad = true;
            rec5 = (u32)ref|((bw&0xFFFFu)<<8);
            if(lane==0) p.frame_bw[f] = bw&0xFFFFu;
        }
        rb.release(it);                                         // after the black/white pass: it reads staged rows 0 and 2
        {
            const u32 bad = __ballot_sync(0xFFFFFFFFu, active&&((!crc_ok)||(is_hdr&&(k!=0))));
            if(bad) frame_bad = true;
        }
        // ---- VideoToDigital per-field rules for a valid line; the previous line of the same field sits two lanes down
        u32 p01 = __shfl_up_sync(0xFFFFFFFFu, w01, 2), p23 = __shfl_up_sync(0xFFFFFFFFu, w23, 2), p45 = __shfl_up_sync(0xFFFFFFFFu, w45, 2);
        bool p_hdr = __shfl_up_sync(0xFFFFFFFFu, is_hdr ? 1 : 0, 2)!=0;
        if(lane<2) { p01 = c01; p23 = c23; p45 = c45; p_hdr = c_hdr; }
        if((k==0)||p_hdr) { p01 = p23 = p45 = 0x10001000u; }       // cleared last_pcm1_line (pcm1line.cpp:56-76)
        u16 wv[6] = { (u16)w0, (u16)w1, (u16)w2, (u16)w3, (u16)w4, (u16)w5 };
        const bool silent = p1_words_almost_silent(wv);
        bool forced_bad = false;
        if(p.line_dup&&!is_hdr)
        {
            if(k==0) forced_bad = true;
            else forced_bad = (packed_diff8(w01, w23, w45, 0u, p01, p23, p45, 0u)<=(P1_BITS/32))&&!silent;
        }
        const int last = rows-2+fld;
        c01 = __shfl_sync(0xFFFFFFFFu, w01, last); c23 = __shfl_sync(0xFFFFFFFFu, w23, last); c45 = __shfl_sync(0xFFFFFFFFu, w45, last);
        c_hdr = __shfl_sync(0xFFFFFFFFu, is_hdr ? 1 : 0, last)!=0;
        // ---- record
        u32 flags, r5 = rec5, r6 = rec6, r7 = picked<<16;
        if(is_hdr)
        {   // PCM1Line::setServHeader: the base fields are cleared, words and picked-bit counts stay
            flags = SDV_LF_CRC_OK|SDV_LF_CRC_OK_IGN;
            r5 = 0; r6 = (u32)(u16)NO_COORD_LEFT|((u32)(u16)NO_COORD_RIGHT<<16); r7 |= (u32)SDV_SRV_HEADER_LINE<<8;
        }
        else
        {
            flags = SDV_LF_CRC_OK_IGN|SDV_LF_BW_SET|SDV_LF_BY_EXT;
            flags |= forced_bad ? SDV_LF_FORCED_BAD : SDV_LF_CRC_OK;
        }
        if(silent) flags |= SDV_LF_ALMOST_SILENT;
        if((!crc_ok)||preset_bad) flags = 0;                    // not decoded here: the chain kernel must not take this record as a hint
        if(active)
        {
            const size_t ridx = (size_t)f*p.H+(size_t)fld*hf+k;
            uint4 *dst = (uint4 *)(p.recs+ridx);
            dst[0] = make_uint4(w01, w23, w45, w6);
            dst[1] = make_uint4(flags<<16, r5, r6, r7);
            if(p.aux) *(uint4 *)(p.aux+ridx) = make_uint4(is_hdr ? 0u : ((u32)ref|((u32)ref<<8)), 0u, 0u, 0u);
        }
        if(b==rb.nbatch-1)
        {
            if(lane==0) p.clean[f] = frame_bad ? 0 : 1;
            frame_bad = false;
        }
    }
}

// ------------------------------------------------------------------------------------------------ the chain
struct P1ChainParams
{
    const u8 *luma; int H, W; size_t stride; int n_frames;
    int mode, line_dup, use_bulk;
    int cont;                       // the call continues the file: the chain starts from *ctx instead of a reset
    const P1Preset *presets; const u8 *clean; const u32 *frame_bw;
    sdv_line_rec *recs; sdv_line_aux *aux;
    P1ChainCtx *ctx;
    unsigned long long *stats;      // [4]: lines decoded by the chain, coordinate searches, frames skipped, reserved
};

// Would a valid line at [cur] pass the coordinate damper against the history entry [old] (3 x PPB, videotodigital.cpp:1315-1361)?
SDV_HD bool p1_within_damper_bits(Coord cur, Coord old, int bits)
{
    u32 psm = (u32)(cur.stop-cur.start);
    psm = (psm*INT_CALC_MULT+(u32)bits/2)/(u32)bits;
    const int lim = (int)(u8)((int)((psm/INT_CALC_MULT)&0xFF)*3);
    const i16 ds = (i16)(cur.start-old.start), de = (i16)(cur.stop-old.stop);
    return !delta_warning(ds, de, lim);
}
SDV_HD bool p1_within_damper(Coord cur, Coord old) { return p1_within_damper_bits(cur, old, P1_BITS); }

// The line object of a hinted line: preset-only decode whose first readPCMdata candidate was valid (STG_INPUT_ALL ->
// readPCMdata -> STG_DATA_OK, binarizer.cpp:774-931,1560-1640), words and picked-bit counts taken from the hint record.
SDV_HD void p1_line_from_hint(P1Line *l, const sdv_line_rec *r, const BinState *b)
{
    p1_clear(l);
    for(int i=0;i<P1L_WORDS;i++) l->words[i] = r->words[i];
    l->calc_crc = l->words[6];
    l->coords = b->def_coord; l->ppb = p1_make_ppb(l->coords);
    l->ref = b->def_ref; l->hyst = r->hyst; l->shift = r->shift;
    l->ref_low = get_low_level(l->ref, l->hyst); l->ref_high = get_high_level(l->ref, l->hyst);
    l->black = b->def_black; l->white = b->def_white; l->bw_set = 1; l->by_ext = 1;
    l->picked_left = (u8)(r->mark_stages&0x0F); l->picked_right = (u8)(r->mark_stages>>4);
    if(p1_words_header(l->words)) p1_set_serv_header(l);
}
// Steady state of the chain inside a field: a valid line decoded with the presets leaves everything but last_words and
// the counters unchanged (the damper sees a history equal to the line's coordinates, the first-line rule is past).
SDV_HD bool p1_chain_steady(const P1ChainCtx *x)
{
    if(x->field_state!=FIELD_INIT) return false;
    if(x->n_last!=COORD_HISTORY_DEPTH) return false;
    for(int i=0;i<COORD_HISTORY_DEPTH;i++) if(!coord_eq(x->last_valid[i], x->bin.def_coord)) return false;
    return true;
}

__global__ void __launch_bounds__(P1L_THREADS) pcm1_chain_kernel(P1ChainParams p)
{
    __shared__ P1Work w;
    __shared__ __align__(16) u8 px[SDV_MAX_W];
    __shared__ int s_skip, s_scr, s_batch;
    __shared__ u16 s_lastw[6];
    __shared__ Coord s_mv, s_mi;
    __shared__ __align__(16) sdv_line_rec s_rec[P1C_CHUNK];
    __shared__ __align__(16) sdv_line_aux s_aux[P1C_CHUNK];
    Cta c = { (int)threadIdx.x, (int)blockDim.x };
    const Geom g = make_geom(p.W);
    // the chain context lives in dynamic shared memory for the run (see pcm16x0_chain_kernel); p.ctx gets a copy
    extern __shared__ __align__(16) u8 chain_dsm[];
    P1ChainCtx *x = (P1ChainCtx *)chain_dsm;
    const int hf = p.H/2;
    if(p.cont) { for(int i=c.tid;i<(int)(sizeof(P1ChainCtx)/4);i+=c.n) ((u32 *)x)[i] = ((const u32 *)p.ctx)[i]; }
    else if(c.tid==0) p1_chain_reset(x, p.mode, p.line_dup);
    if(c.tid==0) { p.stats[0] = p.stats[1] = p.stats[2] = p.stats[3] = 0; }
    __syncthreads();
    const bool opens = !p.cont;         // frame 0 carries the NEW_FILE line
    int f = 0;
    while(f<p.n_frames)
    {
        // ---- look-ahead: how many frames from f on can be taken from the bulk kernel as they are
        if(p.use_bulk)
        {
            if(c.tid==0) s_skip = c.n;
            __syncthreads();
            const int ff = f+c.tid;
            bool ok = false;
            if(ff<p.n_frames)
            {
                const P1Preset ps = p.presets[ff];
                ok = p.clean[ff]&&ps.valid&&coord_valid(ps.coords)&&p1_prescan_runs(p.H, opens&&(ff==0), p.mode);
                if(ok)
                {   // thread 0 checks against the chain's history (carried over on a continuing call), the others against the frame before
                    if(c.tid==0) { for(int i=0;i<x->n_last;i++) if(!p1_within_damper(ps.coords, x->last_valid[i])) ok = false; }
                    else { const P1Preset pv = p.presets[ff-1]; ok = p1_within_damper(ps.coords, pv.coords); }
                }
            }
            if(!ok) atomicMin(&s_skip, c.tid);
            __syncthreads();
            const int n_skip = s_skip;
            __syncthreads();
            if(n_skip>0)
            {
                if(c.tid==0)
                {
                    for(int q=(n_skip>COORD_LONG_HISTORY) ? (n_skip-COORD_LONG_HISTORY) : 0;q<n_skip;q++)
                    {
                        if(x->n_long==COORD_LONG_HISTORY) { for(int k=1;k<COORD_LONG_HISTORY;k++) x->long_valid[k-1] = x->long_valid[k]; x->n_long--; }
                        x->long_valid[x->n_long++] = p.presets[f+q].coords;
                    }
                    const P1Preset ps = p.presets[f+n_skip-1];
                    const u32 bw = p.frame_bw[f+n_skip-1];
                    for(int i=0;i<COORD_HISTORY_DEPTH;i++) x->last_valid[i] = ps.coords;
                    x->n_last = COORD_HISTORY_DEPTH;
                    x->frame_avg = ps.coords; x->prescan_ref = ps.ref;
                    x->bin.def_ref = ps.ref; bin_set_coords(&x->bin, ps.coords); bin_set_bw(&x->bin, (u8)(bw&0xFF), (u8)((bw>>8)&0xFF));
                    x->n_fv = x->n_fi = 0;
                    p1_chain_field_end(x);
                    p.stats[2] += (unsigned long long)n_skip;
                }
                f += n_skip;
                __syncthreads();
                continue;
            }
        }
        // ---- exact sequential decode of frame f
        if(c.tid==0) p1_chain_frame_start(x, p1_prescan_runs(p.H, opens&&(f==0), p.mode), p.presets[f]);
        __syncthreads();
        for(int fld=0;fld<2;fld++)
        {
            int k = 0;
            bool weak_hints = false;            // the last run of hints ended on a line the bulk pass could not take
            while(k<hf)
            {
                // Lines the bulk pass already decoded with exactly the presets the chain holds now (preset-only decode,
                // first candidate valid) only need the chain rules.  A chunk of the field's records is staged in shared
                // memory by the whole block, thread 0 runs ahead over the leading hinted lines, the block stores them back.
                int n_chunk = (hf-k<P1C_CHUNK) ? (hf-k) : P1C_CHUNK;
                const size_t base = (size_t)f*p.H+(size_t)fld*hf+k;
                if(p.use_bulk) for(int i=c.tid;i<2*n_chunk;i+=c.n) ((uint4 *)s_rec)[i] = ((const uint4 *)(p.recs+base))[i];
                __syncthreads();
                {
                    // The hints must have been decoded with the presets the chain holds now.  If the bulk pass used others
                    // (or did not run, or its first-candidate-only hints just proved too weak), the chunk is decoded here,
                    // one line per thread, with the current presets: readPCMdata of the preset-only path with the mode's
                    // hysteresis / pixel-shift limits.
                    const BinState b0 = x->bin;
                    const bool ready = bin_fast_ready(&b0);
                    const sdv_line_rec *r0 = &s_rec[0];
                    const bool match = p.use_bulk&&(((r0->ref==b0.def_ref)&&(r0->data_start==b0.def_coord.start)&&(r0->data_stop==b0.def_coord.stop))
                                                    ||((r0->service_type==SDV_SRV_HEADER_LINE)&&(p.presets[f].ref==b0.def_ref)&&coord_eq(p.presets[f].coords, b0.def_coord)));
                    __syncthreads();
                    if(!ready) n_chunk = 0;
                    else if((!match)||weak_hints)
                    {
                        for(int i=c.tid;i<n_chunk;i+=c.n)
                        {
                            P1Line t;
                            p1_clear(&t);
                            t.ref = b0.def_ref; t.black = b0.def_black; t.white = b0.def_white; t.bw_set = 1;
                            t.coords = b0.def_coord; t.ppb = p1_make_ppb(t.coords);
                            p1_read_pcm(p.luma+((size_t)f*p.H+(size_t)(2*(k+i)+fld))*p.stride, g, p.mode, &t, b0.max_hyst, b0.max_shift);
                            p1_export_line(&t, &s_rec[i], &s_aux[i]);
                        }
                        __syncthreads();
                    }
                }
                if(c.tid==0) { s_skip = 0; s_batch = 0; }
                __syncthreads();
                for(;;)
                {
                    // (A) thread 0, line by line, until the chain is in its steady state (field past its first line, the
                    //     whole coordinate history equal to the presets): there a valid hinted line changes nothing but the
                    //     duplicate-line reference and the counters
                    if(c.tid==0)
                    {
                        int kk = s_skip;
                        s_batch = 0;
                        while(kk<n_chunk)
                        {
                            sdv_line_rec *r = &s_rec[kk];
                            const BinState *b = &x->bin;
                            const bool hdr = (r->service_type==SDV_SRV_HEADER_LINE)||p1_words_header(r->words);
                            if(!((r->flags&SDV_LF_CRC_OK_IGN)&&bin_fast_ready(b)
                                 &&((r->service_type==SDV_SRV_HEADER_LINE)||((b->def_ref==r->ref)&&(b->def_coord.start==r->data_start)&&(b->def_coord.stop==r->data_stop))))) break;
                            if((!hdr)&&p1_chain_steady(x)) { s_batch = 1; break; }
                            P1Line *l = &w.o;
                            p1_line_from_hint(l, r, b);
                            p1_chain_line(x, l);
                            p1_export_line(l, r, &s_aux[kk]);
                            kk++;
                        }
                        p.stats[0] += (unsigned long long)(kk-s_skip); p.stats[3] += (unsigned long long)(kk-s_skip);
                        s_skip = kk;
                        s_scr = n_chunk;
                    }
                    __syncthreads();
                    if(!s_batch) break;
                    // (B) the steady run, one line per thread
                    const int k0 = s_skip;
                    const BinState b = x->bin;
                    for(int i=k0+c.tid;i<n_chunk;i+=c.n)
                    {
                        const sdv_line_rec *r = &s_rec[i];
                        const bool ok = (r->flags&SDV_LF_CRC_OK_IGN)&&(r->service_type==SDV_SRV_NO)&&(!p1_words_header(r->words))
                                        &&(b.def_ref==r->ref)&&(b.def_coord.start==r->data_start)&&(b.def_coord.stop==r->data_stop);
                        if(!ok) atomicMin(&s_scr, i);
                    }
                    __syncthreads();
                    const int k1 = s_scr;               // the run is [k0, k1)
                    u16 pw[6]; P1Line l; bool mine = false; int my_i = 0;
                    // n_chunk <= blockDim: one line per thread
                    {
                        const int i = k0+c.tid;
                        if(i<k1)
                        {
                            mine = true; my_i = i;
                            p1_line_from_hint(&l, &s_rec[i], &b);
                            if(i>k0) for(int q=0;q<6;q++) pw[q] = s_rec[i-1].words[q];
                            else for(int q=0;q<6;q++) pw[q] = x->last_words[q];
                        }
                    }
                    __syncthreads();
                    if(mine)
                    {
                        if(x->line_dup&&(p1_words_diff8(l.words, pw)<=(P1_BITS/32))&&(!p1_words_almost_silent(l.words))) l.forced_bad = 1;
                        if(my_i==(k1-1)) for(int q=0;q<6;q++) s_lastw[q] = l.words[q];
                        const int slot = x->n_fv+(my_i-k0);
                        if(slot<SDV_MAX_H) x->frame_valid[slot] = l.coords;
                        p1_export_line(&l, &s_rec[my_i], &s_aux[my_i]);
                    }
                    __syncthreads();
                    if(c.tid==0)
                    {
                        const int n = k1-k0;
                        if(n>0)
                        {
                            for(int q=0;q<6;q++) x->last_words[q] = s_lastw[q];
                            x->good_in_field += n; x->pcm_in_field += n;
                            x->n_fv = (x->n_fv+n<SDV_MAX_H) ? (x->n_fv+n) : SDV_MAX_H;
                            p.stats[0] += (unsigned long long)n; p.stats[3] += (unsigned long long)n;
                        }
                        s_skip = k1;
                    }
                    __syncthreads();
                    if(k1>=n_chunk) break;
                }
                __syncthreads();
                const int taken = s_skip;
                for(int i=c.tid;i<2*taken;i+=c.n) ((uint4 *)(p.recs+base))[i] = ((const uint4 *)s_rec)[i];
                if(p.aux) for(int i=c.tid;i<taken;i+=c.n) ((uint4 *)(p.aux+base))[i] = ((const uint4 *)s_aux)[i];
                __syncthreads();
                k += taken;
                weak_hints = (taken<n_chunk);
                if((taken==n_chunk)&&(n_chunk>0)) continue;
                if(k>=hf) break;
                const u8 *src = p.luma+((size_t)f*p.H+(size_t)(2*k+fld))*p.stride;
                for(int i=c.tid;i<p.W;i+=c.n) px[i] = __ldg(src+i);
                __syncthreads();
                const BinState b = x->bin;
                const bool search = p1_chain_coord_search(x);
                __syncthreads();
                p1_process_line_cta(c, &w, &b, search, px, g);
                if(c.tid==0)
                {
                    if(w.o.coord_sweeped||w.was_bw_scanned) p.stats[1]++;
                    p1_chain_line(x, &w.o);
                    const size_t ridx = (size_t)f*p.H+(size_t)fld*hf+k;
                    p1_export_line(&w.o, p.recs+ridx, p.aux ? p.aux+ridx : (sdv_line_aux *)0);
                    p.stats[0]++;
                }
                __syncthreads();
                k++;
            }
            if(c.tid==0) p1_chain_field_end(x);
            __syncthreads();
        }
        median_cta(c, x->frame_valid, x->n_fv, &s_mv, &s_scr);
        median_cta(c, x->frame_invalid, x->n_fi, &s_mi, &s_scr);
        if(c.tid==0) p1_chain_frame_end(x, s_mv, s_mi);
        __syncthreads();
        f++;
    }
    for(int i=c.tid;i<(int)(sizeof(P1ChainCtx)/4);i+=c.n) ((u32 *)p.ctx)[i] = ((const u32 *)x)[i];
}

}   // namespace sdv
