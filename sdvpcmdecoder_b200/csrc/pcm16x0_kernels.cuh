// pcm16x0_kernels.cuh -- PCM-16x0 line decode kernels (device only); same plan as pcm1_kernels.cuh:
//
//   pcm16x0_prescan_kernel : prescanCoordinates for every frame at once (right part of four lines per frame, full grid
//                            search each), one thread block per line.
//   pcm1_preset_kernel     : (shared) median of the four results -> per-frame presets.
//   pcm16x0_bulk_kernel    : HBM-bound pass, one warp per frame, one lane per video line = three sub-line records.
//                            With the duplicate-line check on, the reference decodes only the first line of a frame with
//                            the frame's prescan coordinates: that line is forced bad, its right part then presets the
//                            median of the coordinate history (videotodigital.cpp:1427-1516) and every later line follows
//                            it -- so the pass runs with one running coordinate pair G (the file's first frame's; a call
//                            that continues the file reads it from the chain context) plus the
//                            per-frame reference level, and with three black/white measurements per frame (first line,
//                            second line of either field).  Frames decoded completely this way are flagged clean.
//   pcm16x0_chain_kernel   : walks the frames in order; skips runs of clean frames while the chain state is the steady one
//                            the bulk pass assumed, decodes everything else with the exact sequential semantics (hints,
//                            re-hinting and steady-state batches as in pcm1_chain_kernel).
#pragma once
#include "pcm16x0_chain.cuh"
#include "pcm1_kernels.cuh"

namespace sdv {

__global__ void __launch_bounds__(P1S_THREADS, 5) pcm16x0_prescan_kernel(const u8 *luma, int H, int W, size_t stride, int n_frames, int mode, int opens, P1Preset *scan)
{
    __shared__ X0Work w;
    __shared__ __align__(16) u8 px[SDV_MAX_W];
    const int f = blockIdx.x/P1_COORD_CHECK_LINES, idx = blockIdx.x%P1_COORD_CHECK_LINES;
    if(f>=n_frames) return;
    P1Preset r; r.valid = 0; r.ref = 0; r.coords = coord_none(); r.pad[0] = r.pad[1] = 0;
    const int row = p1_prescan_row(H, opens&&(f==0), idx);
    if(row<0) { if(threadIdx.x==0) scan[blockIdx.x] = r; return; }
    const u8 *src = luma+((size_t)f*H+(size_t)row)*stride;
    for(int i=threadIdx.x;i<W;i+=blockDim.x) px[i] = __ldg(src+i);
    if(threadIdx.x==0) w.scan_done = 0;
    __syncthreads();
    Cta c = { (int)threadIdx.x, (int)blockDim.x };
    Geom g = make_geom(W);
    BinState b;
    bin_set_mode(&b, mode);
    b.def_coord = coord_none();
    bin_reset_good(&b);
    x0_process_line_cta(c, &w, &b, X0L_RIGHT, true, px, g);
    if(threadIdx.x==0)
    {
        if(x0_crc_ok(&w.o)) { r.valid = 1; r.coords = w.o.coords; r.ref = w.o.ref; }
        r.pad[0] = w.scan_done;             // VideoLine::scan_done of this line when the frame itself is decoded
        scan[blockIdx.x] = r;
    }
}

// Black/white levels of one staged row (findPCM16X0BW + findBlackWhite tail), by one warp.
__device__ __forceinline__ u32 x0_warp_black_white(const u8 *row, int W, u32 *hist, int lane)
{
    for(int i=lane;i<256;i+=32) hist[i] = 0;
    __syncwarp();
    const int span = W-1, t = span/8;
    int from = span/5;
    for(int i=from+lane;i<from+t;i+=32) atomicAdd(&hist[row[i]], 1u);
    from = t*4+t/2;
    for(int i=from+lane;i<from+t;i+=32) atomicAdd(&hist[row[i]], 1u);
    const int lim = span-span/64;
    for(int i=lim-t+lane;i<lim;i+=32) atomicAdd(&hist[row[i]], 1u);
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
__device__ __forceinline__ bool x0_bw_fits(u32 bw, int ref) { return ((bw>>16)&1u)&&(ref<(int)((bw>>8)&0xFFu))&&(ref>(int)(bw&0xFFu)); }

// bit_i = G_i | (E_i & bit_{i-1}) over a 64-bit MSB-first stream (see resolve_equal_cells).
__device__ __forceinline__ void resolve_equal_cells64(u32 *g, const u32 *ge)
{
    const u32 gr0 = __brev(g[0]), gr1 = __brev(g[1]), er0 = __brev(ge[0]&~g[0]), er1 = __brev(ge[1]&~g[1]);
    const u64 a = ((u64)(gr1|er1)<<32)|(gr0|er0), b = ((u64)gr1<<32)|gr0;
    const u64 s = a+b;
    const u64 cout = (s<a) ? 1ull : 0ull;
    const u64 cin = s^a^b;
    const u64 r = (cin>>1)|(cout<<63);
    g[0] = __brev((u32)r); g[1] = __brev((u32)(r>>32));
}

// Cut-off bit cell counts of a valid line (the forced bit picker only counts): picked_left | picked_right<<4.
__device__ __forceinline__ u32 x0_picked_counts(Ppb pp, int mode, int W)
{
    X0Line t; t.ppb = pp; t.forced_bad = 0; t.calc_crc = 0; for(int i=0;i<X0L_WORDS;i++) t.words[i] = 0;
    x0_pick_cut_bits(&t, mode, X0L_LEFT, W-1, W-1);
    const u32 l = t.picked_left;
    x0_pick_cut_bits(&t, mode, X0L_RIGHT, W-1, W-1);
    return l|((u32)t.picked_right<<4);
}

__global__ void __launch_bounds__(BULK_MAX_WARPS*32, 1) pcm16x0_bulk_kernel(const __grid_constant__ P1BulkParams p)
{
    extern __shared__ __align__(128) u8 dsm[];
    u16 *crc_tab = (u16 *)(dsm+BULK_BAR_BYTES);
    const int warp = threadIdx.x>>5, lane = threadIdx.x&31;
    u32 *hist = (u32 *)(dsm+BULK_BAR_BYTES+512)+warp*256;
    for(int i=threadIdx.x;i<256;i+=blockDim.x) crc_tab[i] = c_crc8[i];
    BulkRing rb(dsm, P1_BULK_HEADER, p.luma, p.H, p.W, p.stride, 0, p.n_frames, p.use_tma, p.warps, p.slot_bytes);
    __syncthreads();
    rb.prime();

    const int hf = p.H/2;
    const int fld = lane&1;
    const int pixel_stop = p.W-1;

    // the running coordinates of the tape (duplicate-line check on): those of the file's first frame
    const P1Preset ps0 = *p.run_g;
    const bool have_g = ps0.valid&&coord_valid(ps0.coords);
    Coord gc = ps0.coords; if(!have_g) { gc.start = 0; gc.stop = (i16)(p.W-1); }
    const Ppb gpp = x0_make_ppb(gc);
    const u32 g_picked = x0_picked_counts(gpp, p.mode, p.W);

    u32 cw[3][2];                               // per part: words of this field's last line in the previous step
    for(int q=0;q<3;q++) cw[q][0] = cw[q][1] = 0;
    bool frame_bad = false, preset_bad = false;
    int ref = 128;
    Ppb fpp = gpp; Coord fc = gc; u32 f_picked = g_picked;      // coordinates of the frame's first line / of the whole frame (no dup check)
    u32 bw0 = 0, bwb = 0, bwc = 0;

    for(long long it=0;it<rb.n_items;it++)
    {
        const BulkItem t = rb.item(it);
        const int f = t.f, b = t.b, r0 = t.r0, rows = t.rows;
        const int k = (r0>>1)+(lane>>1);
        const int frow = r0+lane;
        const bool active = lane<rows;
        if(b==0)
        {
            const P1Preset ps = p.presets[f];
            fc = ps.coords;
            frame_bad = !(ps.valid&&coord_valid(fc))||(p.line_dup&&!have_g);
            preset_bad = frame_bad;
            if(!(ps.valid&&coord_valid(fc))) { fc.start = 0; fc.stop = (i16)(p.W-1); }
            ref = (ps.valid) ? ps.ref : 128;
            fpp = x0_make_ppb(fc);
            f_picked = x0_picked_counts(fpp, p.mode, p.W);
            for(int q=0;q<3;q++) cw[q][0] = cw[q][1] = 0;
        }
        const u8 *stage = rb.acquire(t);
        const u8 *row = stage+(size_t)lane*p.slot_bytes;
        // which coordinates this line is read with: the frame's own without the duplicate-line check; with it only the left
        // and middle part of the frame's first line (its forced-bad middle part already presets the history median)
        const bool own = (!p.line_dup)||(frow==0);
        // ---- 193 bit cells: three parts of 64 with the control bit between the middle and the right one
        u32 g[3][2], ge[3][2];
        bool ctrl[3];
#pragma unroll
        for(int part=0;part<3;part++)
        {
            const bool own_part = own&&((!p.line_dup)||(part<2));
            const u32 psm = own_part ? fpp.psm : gpp.psm, half = own_part ? fpp.half : gpp.half;
            const int ofs = own_part ? fpp.ofs : gpp.ofs;
            {
                int cpos = (int)(((u32)X0L_CTRL_BIT*psm+half)>>7)+ofs;
                cpos = max(0, min(cpos, pixel_stop-1));
                ctrl[part] = row[cpos]>=ref;
            }
#pragma unroll
            for(int w=0;w<2;w++)
            {
                u32 a = 0, c = 0;
#pragma unroll
                for(int j=0;j<32;j++)
                {
                    const int bit = ((part==2) ? 129 : (64*part))+32*w+j;
                    int pos = (int)(((u32)bit*psm+half)>>7)+ofs;
                    pos = max(0, min(pos, pixel_stop-1));
                    const int v = row[pos];
                    a = __funnelshift_l((u32)(ref-v), a, 1);
                    c = __funnelshift_l((u32)(ref-1-v), c, 1);
                }
                g[part][w] = a; ge[part][w] = c;
            }
        }
        bool any_eq = false;
#pragma unroll
        for(int part=0;part<3;part++) any_eq = any_eq||(((ge[part][0]^g[part][0])|(ge[part][1]^g[part][1]))!=0);
        if(__any_sync(0xFFFFFFFFu, any_eq))
        {
#pragma unroll
            for(int part=0;part<3;part++) resolve_equal_cells64(g[part], ge[part]);
        }
        // ---- black/white levels: first line of the frame, second line of either field
        if(b==0)
        {
            bw0 = x0_warp_black_white(stage, p.W, hist, lane);
            if(!x0_bw_fits(bw0, ref)) frame_bad = true;
            if(p.line_dup)
            {
                bwb = x0_warp_black_white(stage+(size_t)2*p.slot_bytes, p.W, hist, lane);
                bwc = x0_warp_black_white(stage+(size_t)3*p.slot_bytes, p.W, hist, lane);
                if(!x0_bw_fits(bwb, ref)||!x0_bw_fits(bwc, ref)) frame_bad = true;
            }
            else bwb = bwc = bw0;
            if(lane==0) p.frame_bw[f] = bwc&0xFFFFu;
        }
        rb.release(it);                                         // after the black/white pass: it reads staged rows 0, 2 and 3
        const u32 bw = (!p.line_dup||(frow==0)) ? bw0 : (((frow&1)&&(frow>=3)) ? bwc : bwb);
        const u32 rec5 = (u32)ref|((bw&0xFFFFu)<<8);
        bool line_ok = true;
#pragma unroll
        for(int part=0;part<3;part++)
        {
            const bool own_part = own&&((!p.line_dup)||(part<2));
            const Coord lc = own_part ? fc : gc;
            const u32 picked = own_part ? f_picked : g_picked;
            const u32 rec6 = (u32)(u16)lc.start|((u32)(u16)lc.stop<<16);
            const u32 g0 = g[part][0], g1 = g[part][1];
            u32 crc = 0xFFFFu;
#pragma unroll
            for(int j=0;j<6;j++)
            {
                const u32 m = (j<4) ? ((g0>>(24-8*j))&0xFFu) : ((g1>>(24-8*(j-4)))&0xFFu);
                crc = ((crc<<8)^crc_tab[((crc>>8)^m)&0xFFu])&0xFFFFu;
            }
            const bool crc_ok = (crc==(g1&0xFFFFu));
            if(!crc_ok) line_ok = false;
            // per-field rules; the previous line of the same field sits two lanes down
            u32 p0 = __shfl_up_sync(0xFFFFFFFFu, g0, 2), p1 = __shfl_up_sync(0xFFFFFFFFu, g1, 2);
            if(lane<2) { p0 = cw[part][0]; p1 = cw[part][1]; }
            if(k==0) { p0 = 0; p1 = 0; }
            u16 wv[3] = { (u16)(g0>>16), (u16)(g0&0xFFFFu), (u16)(g1>>16) };
            const bool silent = x0_words_almost_silent(wv);
            bool forced_bad = false;
            if(p.line_dup)
            {
                if(k==0) forced_bad = true;         // first line of the field: the left part by the rule, the others follow it
                else forced_bad = ((__popc((g0^p0)&0x00FF00FFu)+__popc((g1^p1)&0x00FF0000u))<=(X0L_PART_BITS/32))&&!silent;
            }
            const int last = rows-2+fld;
            cw[part][0] = __shfl_sync(0xFFFFFFFFu, g0, last); cw[part][1] = __shfl_sync(0xFFFFFFFFu, g1, last);
            u32 flags = SDV_LF_CRC_OK_IGN|SDV_LF_BW_SET|SDV_LF_BY_EXT|SDV_LF_COORDS_SET;
            flags |= forced_bad ? SDV_LF_FORCED_BAD : SDV_LF_CRC_OK;
            if(ctrl[part]) flags |= SDV_LF_CONTROL_BIT;
            if(silent) flags |= SDV_LF_ALMOST_SILENT;
            if((!crc_ok)||preset_bad) flags = 0;                // not decoded here: no hint for the chain kernel
            const u32 ms = (part==X0L_LEFT) ? (picked&0x0Fu) : ((part==X0L_RIGHT) ? (picked&0xF0u) : 0u);
            if(active)
            {
                const size_t ridx = ((size_t)f*p.H+(size_t)fld*hf+k)*3+part;
                uint4 *dst = (uint4 *)(p.recs+ridx);
                dst[0] = make_uint4((g0>>16)|(g0<<16), (g1>>16)|(g1<<16), (u32)(3*k+part), 0u);
                dst[1] = make_uint4(flags<<16, rec5, rec6, (ms<<16)|((u32)part<<24));
                if(p.aux) *(uint4 *)(p.aux+ridx) = make_uint4((u32)ref|((u32)ref<<8), 0u, 0u, 0u);
            }
        }
        {
            const u32 bad = __ballot_sync(0xFFFFFFFFu, active&&(!line_ok));
            if(bad) frame_bad = true;
        }
        if(b==rb.nbatch-1)
        {
            if(lane==0) p.clean[f] = frame_bad ? 0 : 1;
            frame_bad = false;
        }
    }
}

// ------------------------------------------------------------------------------------------------ the chain
enum { X0C_CHUNK_LINES = 85 };          // chain kernel: records staged per chunk of lines (3 x 85 sub-lines <= one block of threads)

struct X0ChainParams
{
    const u8 *luma; int H, W; size_t stride; int n_frames;
    int mode, line_dup, use_bulk;
    int cont;                       // the call continues the file: the chain starts from *ctx instead of a reset
    const P1Preset *scan; const P1Preset *presets; const u8 *clean; const u32 *frame_bw;
    sdv_line_rec *recs; sdv_line_aux *aux;
    X0ChainCtx *ctx;
    unsigned long long *stats;
};

// VideoLine::scan_done of a row when the frame itself is decoded: set by the prescan if it searched that row.
__device__ __forceinline__ u8 x0_scan_done_of(const X0ChainParams &p, int f, bool ran, int row)
{
    u8 sd = 0;
    if(ran) for(int idx=0;idx<P1_COORD_CHECK_LINES;idx++) if(p1_prescan_row(p.H, (!p.cont)&&(f==0), idx)==row) sd = p.scan[(size_t)f*P1_COORD_CHECK_LINES+idx].pad[0];
    return sd;
}
// The sub-line object of a hinted sub-line (preset-only decode, first readPCMdata candidate valid).
SDV_HD void x0_line_from_hint(X0Line *l, const sdv_line_rec *r, const BinState *b, int part)
{
    x0_clear(l);
    for(int i=0;i<X0L_WORDS;i++) l->words[i] = r->words[i];
    l->calc_crc = l->words[3];
    l->line_part = (u8)part;
    l->coords = b->def_coord; l->ppb = x0_make_ppb(l->coords);
    l->ref = b->def_ref; l->hyst = r->hyst; l->shift = r->shift;
    l->ref_low = get_low_level(l->ref, l->hyst); l->ref_high = get_high_level(l->ref, l->hyst);
    l->black = b->def_black; l->white = b->def_white; l->bw_set = 1; l->by_ext = 1; l->coords_set = 1;
    l->control_bit = (r->flags&SDV_LF_CONTROL_BIT) ? 1 : 0;
    l->picked_left = (u8)(r->mark_stages&0x0F); l->picked_right = (u8)(r->mark_stages>>4);
}
// Steady state of the chain at the start of a line inside a field (see p1_chain_steady).
SDV_HD bool x0_chain_steady(const X0ChainCtx *x)
{
    if(x->field_state!=FIELD_INIT) return false;
    if(x->n_last!=COORD_HISTORY_DEPTH*3) return false;
    for(int i=0;i<COORD_HISTORY_DEPTH*3;i++) if(!coord_eq(x->last_valid[i], x->bin.def_coord)) return false;
    return true;
}

__global__ void __launch_bounds__(P1L_THREADS) pcm16x0_chain_kernel(X0ChainParams p)
{
    __shared__ X0Work w;
    __shared__ __align__(16) u8 px[SDV_MAX_W];
    __shared__ int s_skip, s_scr, s_batch;
    __shared__ u16 s_lastw[3][3];
    __shared__ Coord s_mv, s_mi;
    __shared__ __align__(16) sdv_line_rec s_rec[3*X0C_CHUNK_LINES];
    __shared__ __align__(16) sdv_line_aux s_aux[3*X0C_CHUNK_LINES];
    Cta c = { (int)threadIdx.x, (int)blockDim.x };
    const Geom g = make_geom(p.W);
    // the chain context (thread 0 reads and writes it on every sub-line) lives in dynamic shared memory for the run; p.ctx gets a copy
    extern __shared__ __align__(16) u8 chain_dsm[];
    X0ChainCtx *x = (X0ChainCtx *)chain_dsm;
    const int hf = p.H/2;
    const int depth = COORD_HISTORY_DEPTH*3;
    if(p.cont) { for(int i=c.tid;i<(int)(sizeof(X0ChainCtx)/4);i+=c.n) ((u32 *)x)[i] = ((const u32 *)p.ctx)[i]; }
    else if(c.tid==0) { x0_chain_reset(x, p.mode, p.line_dup); x->run_g = p.presets[0]; }
    if(c.tid==0) { p.stats[0] = p.stats[1] = p.stats[2] = p.stats[3] = 0; }
    __syncthreads();
    const bool opens = !p.cont;         // frame 0 carries the NEW_FILE line
    const P1Preset ps0 = x->run_g;      // the running pair G the bulk pass decoded with
    int f = 0;
    while(f<p.n_frames)
    {
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
                if(ok&&p.line_dup)
                {   // steady state the bulk pass assumed: the whole coordinate history equals the running pair G (only the
                    // file's first frame is decoded with G as its own prescan coordinates)
                    if((c.tid==0)&&((ff>0)||!opens))
                    {
                        if(x->n_last!=depth) ok = false;
                        for(int i=0;ok&&(i<x->n_last);i++) if(!coord_eq(x->last_valid[i], ps0.coords)) ok = false;
                    }
                }
                else if(ok)
                {
                    if(c.tid==0) { for(int i=0;i<x->n_last;i++) if(!p1_within_damper_bits(ps.coords, x->last_valid[i], X0L_BITS)) ok = false; }
                    else { const P1Preset pv = p.presets[ff-1]; ok = p1_within_damper_bits(ps.coords, pv.coords, X0L_BITS); }
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
                        x->long_valid[x->n_long++] = p.line_dup ? ps0.coords : p.presets[f+q].coords;
                    }
                    const P1Preset ps = p.presets[f+n_skip-1];
                    const Coord run = p.line_dup ? ps0.coords : ps.coords;
                    const u32 bw = p.frame_bw[f+n_skip-1];
                    for(int i=0;i<depth;i++) x->last_valid[i] = run;
                    x->n_last = depth;
                    x->frame_avg = run; x->prescan_ref = ps.ref;
                    x->bin.def_ref = ps.ref; bin_set_coords(&x->bin, run); bin_set_bw(&x->bin, (u8)(bw&0xFF), (u8)((bw>>8)&0xFF));
                    x->n_fv = x->n_fi = 0;
                    x0_chain_field_end(x);
                    x->force_bad_line = 0;
                    p.stats[2] += (unsigned long long)n_skip;
                }
                f += n_skip;
                __syncthreads();
                continue;
            }
        }
        // ---- exact sequential decode of frame f
        const bool ran = p1_prescan_runs(p.H, opens&&(f==0), p.mode);
        if(c.tid==0) x0_chain_frame_start(x, ran, p.presets[f]);
        __syncthreads();
        for(int fld=0;fld<2;fld++)
        {
            int k = 0, part0 = 0;               // next sub-line to decode: line k of the field, part part0
            bool weak_hints = false;            // the last run of hints ended on a sub-line the bulk pass could not take
            while(k<hf)
            {
                // Sub-lines the bulk pass decoded with exactly the presets the chain holds now only need the chain rules:
                // a chunk of records is staged in shared memory, thread 0 runs ahead over the leading hinted sub-lines.
                int n_chunk = 0;
                const size_t base = ((size_t)f*p.H+(size_t)fld*hf+k)*3;
                if(part0==0)
                {
                    n_chunk = 3*(((hf-k)<X0C_CHUNK_LINES) ? (hf-k) : X0C_CHUNK_LINES);
                    if(p.use_bulk) for(int i=c.tid;i<2*n_chunk;i+=c.n) ((uint4 *)s_rec)[i] = ((const uint4 *)(p.recs+base))[i];
                }
                __syncthreads();
                if(n_chunk>0)
                {
                    // hints decoded with other presets than the chain holds now (or none at all, or first-candidate-only hints
                    // that just proved too weak): decode the chunk here, one sub-line per thread, readPCMdata of the preset-only
                    // path with the mode's hysteresis / pixel-shift limits
                    const BinState b0 = x->bin;
                    const bool ready = bin_fast_ready(&b0);
                    const sdv_line_rec *r0 = &s_rec[0];
                    const bool match = p.use_bulk&&(r0->ref==b0.def_ref)&&(r0->data_start==b0.def_coord.start)&&(r0->data_stop==b0.def_coord.stop);
                    __syncthreads();
                    if(!ready) n_chunk = 0;
                    else if((!match)||weak_hints)
                    {
                        for(int i=c.tid;i<n_chunk;i+=c.n)
                        {
                            const int kl = i/3, part = i-3*kl;
                            X0Line t;
                            x0_clear(&t);
                            t.line_part = (u8)part;
                            t.ref = b0.def_ref; t.black = b0.def_black; t.white = b0.def_white; t.bw_set = 1;
                            t.coords = b0.def_coord; t.ppb = x0_make_ppb(t.coords);
                            x0_read_pcm(p.luma+((size_t)f*p.H+(size_t)(2*(k+kl)+fld))*p.stride, g, p.mode, part, &t, b0.max_hyst, b0.max_shift);
                            x0_export_line(&t, &s_rec[i], &s_aux[i]);
                        }
                        __syncthreads();
                    }
                }
                if(c.tid==0) { s_skip = 0; s_batch = 0; }
                __syncthreads();
                for(;;)
                {
                    // (A) thread 0, sub-line by sub-line, until the chain is in its steady state at the start of a line
                    if(c.tid==0)
                    {
                        int q = s_skip;
                        s_batch = 0;
                        while(q<n_chunk)
                        {
                            const int kl = q/3, part = q-3*kl;
                            sdv_line_rec *r = &s_rec[q];
                            const BinState *b = &x->bin;
                            if(!((r->flags&SDV_LF_CRC_OK_IGN)&&bin_fast_ready(b)&&(b->def_ref==r->ref)
                                 &&(b->def_coord.start==r->data_start)&&(b->def_coord.stop==r->data_stop))) break;
                            if((part==0)&&x0_chain_steady(x)) { s_batch = 1; break; }
                            if(part==0)
                            {
                                w.scan_done = x0_scan_done_of(p, f, ran, 2*(k+kl)+fld);
                                x0_chain_line_start(x);
                            }
                            X0Line *l = &w.o;
                            x0_line_from_hint(l, r, b, part);
                            x0_chain_subline(x, l, w.scan_done!=0);
                            x0_export_line(l, r, &s_aux[q]);
                            q++;
                        }
                        p.stats[0] += (unsigned long long)(q-s_skip); p.stats[3] += (unsigned long long)(q-s_skip);
                        s_skip = q;
                        s_scr = n_chunk;
                    }
                    __syncthreads();
                    if(!s_batch) break;
                    // (B) the steady run, one sub-line per thread (n_chunk <= blockDim)
                    const int q0 = s_skip;              // a left part
                    const BinState b = x->bin;
                    {
                        const int i = q0+c.tid;
                        if(i<n_chunk)
                        {
                            const sdv_line_rec *r = &s_rec[i];
                            const bool ok = (r->flags&SDV_LF_CRC_OK_IGN)&&(b.def_ref==r->ref)&&(b.def_coord.start==r->data_start)&&(b.def_coord.stop==r->data_stop);
                            if(!ok) atomicMin(&s_scr, i);
                        }
                    }
                    __syncthreads();
                    const int q1 = s_scr;               // the run is [q0, q1)
                    u16 pw[3]; X0Line l; bool mine = false; int my_i = 0, my_part = 0;
                    {
                        const int i = q0+c.tid;
                        if(i<q1)
                        {
                            mine = true; my_i = i; my_part = (i-q0)%3;
                            x0_line_from_hint(&l, &s_rec[i], &b, my_part);
                            if(i-3>=q0) for(int t=0;t<3;t++) pw[t] = s_rec[i-3].words[t];
                            else for(int t=0;t<3;t++) pw[t] = x->last_words[my_part][t];
                        }
                    }
                    __syncthreads();
                    if(mine)
                    {
                        l.queue_order = (u16)(x->line_in_field+(my_i-q0));
                        if(x->line_dup&&(x0_words_diff8(l.words, pw)<=(X0L_PART_BITS/32))&&(!x0_words_almost_silent(l.words))) l.forced_bad = 1;
                        if(my_i+3>=q1) for(int t=0;t<3;t++) s_lastw[my_part][t] = l.words[t];
                        const int slot = x->n_fv+(my_i-q0);
                        if(slot<SDV_MAX_H*3) x->frame_valid[slot] = l.coords;
                        x0_export_line(&l, &s_rec[my_i], &s_aux[my_i]);
                    }
                    __syncthreads();
                    if(c.tid==0)
                    {
                        const int n = q1-q0;
                        if(n>0)
                        {
                            for(int pt=0;pt<3;pt++) if(pt<n) for(int t=0;t<3;t++) x->last_words[pt][t] = s_lastw[pt][t];
                            x->good_in_field += n; x->pcm_in_field += n; x->line_in_field += n;
                            x->n_fv = (x->n_fv+n<SDV_MAX_H*3) ? (x->n_fv+n) : SDV_MAX_H*3;
                            p.stats[0] += (unsigned long long)n; p.stats[3] += (unsigned long long)n;
                            // the line the run stops in keeps going through (A) / the whole block: its per-line state
                            w.scan_done = x0_scan_done_of(p, f, ran, 2*(k+(q1-1)/3)+fld);
                            x->force_bad_line = 0;
                        }
                        s_skip = q1;
                    }
                    __syncthreads();
                    if(q1>=n_chunk) break;
                }
                __syncthreads();
                const int taken = s_skip;
                for(int i=c.tid;i<2*taken;i+=c.n) ((uint4 *)(p.recs+base))[i] = ((const uint4 *)s_rec)[i];
                if(p.aux) for(int i=c.tid;i<taken;i+=c.n) ((uint4 *)(p.aux+base))[i] = ((const uint4 *)s_aux)[i];
                __syncthreads();
                k += taken/3; part0 += taken%3;         // part0 was 0 whenever a chunk was taken
                if(n_chunk>0) weak_hints = (taken<n_chunk);
                if((taken==n_chunk)&&(n_chunk>0)) continue;
                if(k>=hf) break;
                // ---- the whole block on line k, from part part0 on
                const int row = 2*k+fld;
                const u8 *src = p.luma+((size_t)f*p.H+(size_t)row)*p.stride;
                for(int i=c.tid;i<p.W;i+=c.n) px[i] = __ldg(src+i);
                if((c.tid==0)&&(part0==0))
                {
                    w.scan_done = x0_scan_done_of(p, f, ran, row);
                    x0_chain_line_start(x);
                }
                __syncthreads();
                for(int part=part0;part<3;part++)
                {
                    const BinState b = x->bin;
                    const bool search = x0_chain_coord_search(x);
                    __syncthreads();
                    x0_process_line_cta(c, &w, &b, part, search, px, g);
                    if(c.tid==0)
                    {
                        x0_chain_subline(x, &w.o, w.scan_done!=0);
                        const size_t ridx = ((size_t)f*p.H+(size_t)fld*hf+k)*3+part;
                        x0_export_line(&w.o, p.recs+ridx, p.aux ? p.aux+ridx : (sdv_line_aux *)0);
                        p.stats[0]++;
                    }
                    __syncthreads();
                }
                k++; part0 = 0;
            }
            if(c.tid==0) x0_chain_field_end(x);
            __syncthreads();
        }
        median_cta(c, x->frame_valid, x->n_fv, &s_mv, &s_scr);
        median_cta(c, x->frame_invalid, x->n_fi, &s_mi, &s_scr);
        if(c.tid==0) x0_chain_frame_end(x, s_mv, s_mi);
        __syncthreads();
        f++;
    }
    for(int i=c.tid;i<(int)(sizeof(X0ChainCtx)/4);i+=c.n) ((u32 *)p.ctx)[i] = ((const u32 *)x)[i];
}

}   // namespace sdv
