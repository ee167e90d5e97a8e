// sdv_kernels.cu -- the C ABI (include/sdvpcm.h), the launch logic and the STC-007 kernels that are not in a header.
//
// Kernels (device code lives in the .cuh files named):
//   stc007_bulk_kernel   (stc007_bulk.cuh)  : the HBM-bound pass.  Persistent, one lane per video line, 32 consecutive
//                          frame rows per warp step through a per-warp two-stage ring of 1-D bulk copies (cp.async.bulk +
//                          mbarrier); the 128 bit cells are shifted into two registers per lane ("pixel > ref", "pixel >=
//                          ref"), cells on the reference level resolved as a 128-bit carry chain, CRCC by a byte table,
//                          the per-field VideoToDigital rules (first line of a field, duplicate line) in registers.
//   stc007_chain_kernel  (here; stc007_line.cuh, stc007_chain.cuh) : exact sequential semantics for everything the bulk
//                          pass cannot take: the first frame and every frame with a line that fails the preset decode.
//                          One block (or one block per segment); warps look ahead with the preset decode, the whole block
//                          runs the full Binarizer on a failing line, thread 0 advances the chain.
//   stc007_deint_kernel  (here; stc007_deint.cuh) : one thread per data block (two adjacent blocks per lane, packed in
//                          16-bit halves, in the standard setting), per-warp tiles staged through shared
//                          memory, P/Q correction in registers, samples + flags out; broken_window_kernel for the
//                          128-block unsafe windows; stc007_seam_kernel for the field-seam padding sweep.
//   pcm1_* / pcm16x0_*   (pcm1_kernels.cuh, pcm16x0_kernels.cuh, pcm1_stitch.cuh, pcm16x0_stitch.cuh, *_deint.cuh) :
//                          prescan (grid coordinate search), per-frame presets, bulk pass, chain, frame assembly and
//                          deinterleave for PCM-1 and PCM-16x0.
#include <cuda_runtime.h>
#include <stdio.h>
#include <new>
#include <vector>
#include <algorithm>
#include <memory>
#include "stc007_chain.cuh"
#include "stc007_deint.cuh"
#include "stc007_stitch_host.h"
#include "stc007_bulk.cuh"
#include <unordered_map>
#include <mutex>
#include <chrono>
#include "pcm1_deint.cuh"
#include "pcm16x0_deint.cuh"
#include "pcm1_kernels.cuh"
#include "pcm1_stitch.cuh"
#include "pcm16x0_kernels.cuh"
#include "pcm16x0_stitch.cuh"
#include "pcm16x0_stitch_host.h"
#include "chain_state.cuh"

namespace sdv {

// ------------------------------------------------------------------------------------------------ CRC by linearity
// crc(message) = XOR of c_crc_bit[i] over the set message bits i (stream order) XOR c_crc_zero.
__constant__ u16 c_crc_bit[112];
__constant__ u16 c_crc_zero;

struct FastPos { int p0, p1, p2, p3; u32 t0, t1, t2, t3; };

__device__ __forceinline__ FastPos make_fast_pos(Coord coords, int W, int lane)
{
    FastPos f;
    Ppb ppb = make_ppb(coords);
    f.p0 = pixel_of_bit(ppb, lane, 0, W-1);
    f.p1 = pixel_of_bit(ppb, lane+32, 0, W-1);
    f.p2 = pixel_of_bit(ppb, lane+64, 0, W-1);
    f.p3 = pixel_of_bit(ppb, lane+96, 0, W-1);
    f.t0 = c_crc_bit[lane]; f.t1 = c_crc_bit[lane+32]; f.t2 = c_crc_bit[lane+64];
    f.t3 = (lane<16) ? c_crc_bit[lane+96] : 0;
    return f;
}

// 14-bit word k (k = 0..7) or the 16-bit CRCC (k = 8) from the 128 line bits (bit i of the line = bit i&31 of b[i>>5]).
template<int K>
__device__ __forceinline__ u32 extract_word(u32 b0, u32 b1, u32 b2, u32 b3)
{
    constexpr int o = 14*K, idx = o>>5, off = o&31;
    u32 lo = (idx==0) ? b0 : ((idx==1) ? b1 : ((idx==2) ? b2 : b3));
    u32 hi = (idx==0) ? b1 : ((idx==1) ? b2 : ((idx==2) ? b3 : 0u));
    u32 v = __funnelshift_r(lo, hi, off);
    if(K<8) return __brev(v&0x3FFFu)>>18;
    return __brev(v&0xFFFFu)>>16;
}

struct FastOut { u32 w01, w23, w45, w67, crc_read; bool crc_ok; };

// Preset decode of one row by one warp: bit cells with hysteresis depth 0 (low = high = ref):
// bit_i = (px_i > ref) | ((px_i == ref) & bit_{i-1}), i.e. the carry chain of (G|E) + G.
__device__ __forceinline__ FastOut warp_fast_decode(u32 v0, u32 v1, u32 v2, u32 v3, u32 ref, const FastPos &fp, int lane)
{
    const u32 full = 0xFFFFFFFFu;
    u32 g0 = __ballot_sync(full, v0>ref), e0 = __ballot_sync(full, v0==ref);
    u32 g1 = __ballot_sync(full, v1>ref), e1 = __ballot_sync(full, v1==ref);
    u32 g2 = __ballot_sync(full, v2>ref), e2 = __ballot_sync(full, v2==ref);
    u32 g3 = __ballot_sync(full, v3>ref), e3 = __ballot_sync(full, v3==ref);
    u32 b0 = g0, b1 = g1, b2 = g2, b3 = g3;
    if((e0|e1|e2|e3)!=0)
    {   // rare: some cell sits exactly on the reference level
        u64 alo = ((u64)(g1|e1)<<32)|(g0|e0), ahi = ((u64)(g3|e3)<<32)|(g2|e2);
        u64 blo = ((u64)g1<<32)|g0, bhi = ((u64)g3<<32)|g2;
        u64 slo = alo+blo;
        u64 cy = (slo<alo) ? 1ull : 0ull;
        u64 shi = ahi+bhi+cy;
        u64 cout = ((shi<ahi)||(cy&&(shi==ahi))) ? 1ull : 0ull;
        u64 clo = slo^alo^blo, chi = shi^ahi^bhi;          // carry INTO each bit
        u64 rlo = (clo>>1)|(chi<<63), rhi = (chi>>1)|(cout<<63);    // carry OUT of each bit = the decoded bit
        b0 = (u32)rlo; b1 = (u32)(rlo>>32); b2 = (u32)rhi; b3 = (u32)(rhi>>32);
    }
    FastOut o;
    u32 w0 = extract_word<0>(b0, b1, b2, b3), w1 = extract_word<1>(b0, b1, b2, b3);
    u32 w2 = extract_word<2>(b0, b1, b2, b3), w3 = extract_word<3>(b0, b1, b2, b3);
    u32 w4 = extract_word<4>(b0, b1, b2, b3), w5 = extract_word<5>(b0, b1, b2, b3);
    u32 w6 = extract_word<6>(b0, b1, b2, b3), w7 = extract_word<7>(b0, b1, b2, b3);
    o.crc_read = extract_word<8>(b0, b1, b2, b3);
    o.w01 = w0|(w1<<16); o.w23 = w2|(w3<<16); o.w45 = w4|(w5<<16); o.w67 = w6|(w7<<16);
    u32 x = (((b0>>lane)&1u) ? fp.t0 : 0u)^(((b1>>lane)&1u) ? fp.t1 : 0u)^(((b2>>lane)&1u) ? fp.t2 : 0u)^(((b3>>lane)&1u) ? fp.t3 : 0u);
    u32 crc = __reduce_xor_sync(full, x)^(u32)c_crc_zero;
    o.crc_ok = (crc==o.crc_read);
    return o;
}

// ------------------------------------------------------------------------------------------------ chain kernel
struct ChainParams
{
    const u8 *luma; int H, W; size_t stride;
    int f_begin, n_frames, max_frames;
    sdv_line_rec *recs; sdv_line_aux *aux;
    ChainCtx *ctx;
    const u8 *clean; int have_spec; u8 spec_ref; Coord spec_coords;
    int reset, mode, line_dup;      // reset = 1: start of a file (chain_reset)
    int segments;                   // > 1: the tape is cut into that many independent files, one per thread block (no hand-off)
    // relay mode (relay_len > 0): frames [f_begin, n_frames) in pieces of relay_len frames, one per thread block, for ONE file.
    // Block 0 continues from the true chain state (ctx[0] as the launch finds it).  Every other block builds its own state by
    // decoding the relay_warm frames before its piece (records not kept), its long coordinate history seeded from the
    // per-frame coordinate medians of an earlier pass (fmed_in); start_ctx[b] = its state at the head of the piece, ctx[b] =
    // at the tail.  The host keeps piece b only if start_ctx[b] equals ctx[b-1], i.e. if the guess was the true state.
    int relay_len, relay_warm;
    int plain;                      // 1: run max_frames frames whatever the chain's state (no hand-over to the bulk pass)
    int cont;                       // 1: frame 0 does not open a file (the call continues the file of the call before)
    const Coord *fmed_in; Coord *fmed_out;      // per-frame median of the valid lines' coordinates (what chain_frame_end pushes)
    ChainCtx *start_ctx;
    sdv_line_rec *warm_scratch;                 // CHAIN_BATCH records per block: where warm-up frames put their records
    const int *relay_list;                      // redo round: block i decodes piece relay_list[i] from ctx[piece-1] (the end state of the piece before)
    ChainSnap *snaps;                           // relay mode: the chain state at the head of every kept frame, as last decoded
};

enum { CHAIN_BATCH = 320 };

// CHAIN_THREADS = 1024 for the single sequential chain of a file (everything parallel inside a line gets the whole SM);
// 256 in segment mode, where four independent chains share an SM and fill each other's serial stretches.
template<int CHAIN_THREADS>
__global__ void __launch_bounds__(CHAIN_THREADS, (CHAIN_THREADS==1024) ? 1 : 4) stc007_chain_kernel(ChainParams p)
{
    __shared__ Work w;
    __shared__ BinState s_bin;
    __shared__ __align__(16) u8 row[SDV_MAX_W];
    // look-ahead results of up to one field; they alias the sweep's trial table (never live at the same time)
    static_assert(sizeof(w.sweep_trials)>=CHAIN_BATCH*(sizeof(FastRes)+sizeof(FastPlan)), "look-ahead batch does not fit");
    FastRes *fr = (FastRes *)w.sweep_trials;
    FastPlan *plan = (FastPlan *)(fr+CHAIN_BATCH);
    __shared__ int s_adv, s_stop;
    __shared__ Coord s_med[2];
    const int tid = threadIdx.x, warp = tid>>5, lane = tid&31;
    const Cta c = { tid, CHAIN_THREADS };
    const Geom g = make_geom(p.W);
    // the chain context lives in shared memory while the kernel runs (thread 0 touches it for every line)
    __shared__ __align__(16) ChainCtx sx;
    const bool relay = p.relay_len>0;
    const bool redo = relay&&(p.relay_list!=NULL)&&(p.fmed_in==NULL);      // (a list with medians to seed from: the listed pieces are guessed afresh)
    const int piece = (relay&&p.relay_list) ? p.relay_list[blockIdx.x] : (int)blockIdx.x;
    ChainCtx *gctx = p.ctx+piece;
    const bool load_ctx = relay ? (redo||(piece==0)) : (!p.reset);
    {
        const ChainCtx *src = redo ? (p.ctx+(piece-1)) : gctx;
        if(load_ctx) for(int i=tid;i<(int)(sizeof(ChainCtx)/4);i+=CHAIN_THREADS) ((u32 *)&sx)[i] = ((const u32 *)src)[i];
        else if(tid==0) chain_reset(&sx, p.mode, p.line_dup);
    }
    __syncthreads();
    ChainCtx *x = &sx;
    const int hf = p.H/2;
    const bool seg_mode = p.segments>1;
    int f_first = seg_mode ? (int)((long long)blockIdx.x*p.n_frames/p.segments) : (p.cont ? -1 : 0);       // frame that opens the file
    int f_end = seg_mode ? (int)((long long)(blockIdx.x+1)*p.n_frames/p.segments) : p.n_frames;
    int f = seg_mode ? f_first : p.f_begin, nproc = 0, stable = 0, look = CHAIN_THREADS/32;
    int f_keep = f;                 // first frame whose records are kept (relay: the frames before it only build state)
    if(relay)
    {
        f_keep = p.f_begin+piece*p.relay_len;
        f_end = (f_keep+p.relay_len<p.n_frames) ? (f_keep+p.relay_len) : p.n_frames;
        f = f_keep; f_first = -1;
        if((piece>0)&&!redo)
        {
            f = (f_keep>p.relay_warm) ? (f_keep-p.relay_warm) : 0;
            if(f==0) f_first = 0;                                   // reaches back to the head of the file: nothing to guess
            else if((tid==0)&&p.fmed_in)
            {   // the last 16 valid frame medians before the warm-up, oldest first (long_coord_list)
                Coord tmp[COORD_LONG_HISTORY]; int n = 0;
                for(int q=f-1;(q>=0)&&(q>=f-4*COORD_LONG_HISTORY)&&(n<COORD_LONG_HISTORY);q--) { const Coord m = p.fmed_in[q]; if(coord_valid(m)) tmp[n++] = m; }
                for(int i=0;i<n;i++) x->long_valid[i] = tmp[n-1-i];
                x->n_long = n;
            }
        }
        if(f_keep>=p.n_frames) return;
    }
    if(f>=f_end) return;
    sdv_line_rec *const scratch = p.warm_scratch ? (p.warm_scratch+(size_t)piece*CHAIN_BATCH) : (sdv_line_rec *)0;
    for(;;)
    {
        const bool warming = relay&&(f<f_keep);
        if(relay&&(f==f_keep)&&(piece>0))
        {   // head of the piece: this is the state the piece is decoded from
            __syncthreads();
            if(tid==0) { x->lines_chain = x->lines_chain_fast = x->lines_swept = 0; }
            __syncthreads();
            ChainCtx *sc = p.start_ctx+piece;
            for(int i=tid;i<(int)(sizeof(ChainCtx)/4);i+=CHAIN_THREADS) ((u32 *)sc)[i] = ((const u32 *)&sx)[i];
            __syncthreads();
        }
        if(relay&&!warming&&p.snaps)
        {   // A piece decoded again meets, sooner or later, the states it went through the first time (the chain forgets):
            // from that frame on everything it would write is already there, its old end state included.
            if(tid==0)
            {
                ChainSnap sn; chain_snap(x, &sn);
                s_stop = (redo&&(f>f_keep)&&chain_snap_equal(&sn, &p.snaps[f])) ? 4 : 0;
                if(!s_stop) p.snaps[f] = sn;
            }
            c.sync();
            if(s_stop==4) return;
        }
        if(tid==0) { chain_frame_start(x, f==f_first); s_bin = x->bin; }
        const u8 *frame = p.luma+(size_t)f*p.H*p.stride;
        for(int fld=0;fld<2;fld++)
        {
            int k = 0;
            while(k<hf)
            {
                c.sync();
                const bool ready = bin_fast_ready(&s_bin);
                bool slow = !ready;
                if(ready)
                {   // look ahead: preset decode of the next lines, one per warp
                    // one line per warp to begin with; the look-ahead doubles while whole batches are taken (clean stretches) and
                    // falls back after a line that fails the preset decode -- on a damaged tape the presets change every few
                    // lines, and everything decoded beyond the failing line would be thrown away
                    const int nb = (hf-k<look) ? (hf-k) : look;
                    const FastPos fp = make_fast_pos(s_bin.def_coord, p.W, lane);
                    for(int i=warp;i<nb;i+=CHAIN_THREADS/32)
                    {
                        const u8 *r = frame+(size_t)(2*(k+i)+fld)*p.stride;
                        FastOut o = warp_fast_decode(__ldg(r+fp.p0), __ldg(r+fp.p1), __ldg(r+fp.p2), __ldg(r+fp.p3), s_bin.def_ref, fp, lane);
                        if(lane==0)
                        {
                            FastRes *q = &fr[i];
                            q->words[0] = (u16)o.w01; q->words[1] = (u16)(o.w01>>16); q->words[2] = (u16)o.w23; q->words[3] = (u16)(o.w23>>16);
                            q->words[4] = (u16)o.w45; q->words[5] = (u16)(o.w45>>16); q->words[6] = (u16)o.w67; q->words[7] = (u16)(o.w67>>16);
                            q->words[8] = (u16)o.crc_read; q->ok = o.crc_ok ? 1 : 0;
                        }
                    }
                    // the leading valid lines of the batch are finished in parallel (they leave the presets unchanged)
                    const size_t ridx0 = (size_t)f*p.H+(size_t)fld*hf+k;
                    const int taken = chain_fast_batch(c, x, fr, nb, plan, &s_adv, warming ? scratch : (p.recs+ridx0),
                                                       (p.aux&&!warming) ? p.aux+ridx0 : (sdv_line_aux *)0);
                    k += taken;
                    slow = taken<nb;
                    look = slow ? (CHAIN_THREADS/32) : ((2*look<CHAIN_BATCH) ? (2*look) : CHAIN_BATCH);
                }
                if(slow&&(k<hf))
                {   // full Binarizer on this line by the whole block
                    const u8 *r = frame+(size_t)(2*k+fld)*p.stride;
                    c.sync();
                    for(int i=tid;i<p.W;i+=CHAIN_THREADS) row[i] = __ldg(r+i);
                    c.sync();
                    process_line_cta(c, &w, &s_bin, row, g);
                    if(tid==0)
                    {
                        if(w.do_sweep) x->lines_swept++;
                        chain_line(x, &w.o);
                        const size_t ridx = (size_t)f*p.H+(size_t)fld*hf+k;
                        export_line(&w.o, warming ? scratch : (p.recs+ridx), (p.aux&&!warming) ? p.aux+ridx : (sdv_line_aux *)0);
                        s_bin = x->bin;
                        x->lines_chain++;
                    }
                    k++;
                }
            }
            c.sync();
            if(tid==0) { chain_field_end(x); }
        }
        c.sync();
        median_cta(c, x->frame_valid, x->n_fv, &s_med[0], &s_adv);
        median_cta(c, x->frame_invalid, x->n_fi, &s_med[1], &s_adv);
        if(tid==0)
        {
            if(p.fmed_out&&!warming) p.fmed_out[f] = s_med[0];
            chain_frame_end(x, s_med[0], s_med[1]);
            s_bin = x->bin;
            int stop = ((f+1>=f_end)||((!relay)&&(nproc+1>=p.max_frames))) ? 1 : 0, st = 0;
            if((!seg_mode)&&(!relay)&&(!p.plain)&&(f+1<f_end)&&chain_is_stable(x))
            {
                const bool match = p.have_spec&&(p.spec_ref==x->bin.def_ref)&&coord_eq(p.spec_coords, x->bin.def_coord);
                if(match) { if(p.clean[2*(f+1)]&&p.clean[2*(f+1)+1]) { stop = 1; st = 1; } }
                else { stop = 1; st = 1; }
            }
            s_stop = stop|(st<<1);
        }
        c.sync();
        f++; nproc++;
        if(s_stop&1) { stable = s_stop>>1; break; }
    }
    if(tid==0) { x->next_frame = f; x->stable = stable; x->first_unclean = p.n_frames; }
    __syncthreads();
    for(int i=tid;i<(int)(sizeof(ChainCtx)/4);i+=CHAIN_THREADS) ((u32 *)gctx)[i] = ((const u32 *)&sx)[i];
}

__global__ void set_int_kernel(int *p, int v) { *p = v; }
// Relay mode: piece b was decoded from the true state iff its start state equals the end state of piece b-1.
__global__ void chain_verify_kernel(const ChainCtx *start_ctx, const ChainCtx *end_ctx, int n, u8 *ok)
{
    const int b = blockIdx.x*blockDim.x+threadIdx.x;
    if(b>=n) return;
    ok[b] = (b==0) ? 1 : (chain_state_equal(&start_ctx[b], &end_ctx[b-1]) ? 1 : 0);
}
// First guess of the per-frame coordinate medians: the ones the true chain state remembers (long_coord_list) for the frames
// before f_begin, and the newest of them for every frame from f_begin on -- the history feeds itself (a frame's lines
// inherit the preset coordinates, which come from the median of the history), so it rarely moves.
__global__ void seed_fmed_kernel(const ChainCtx *x, Coord *fmed, int f_begin, int n_frames)
{
    const int n = x->n_long;
    const int i = blockIdx.x*blockDim.x+threadIdx.x;
    if(i>=n_frames) return;
    Coord v = coord_none();
    if(i>=f_begin) { if(n>0) v = x->long_valid[n-1]; }
    else if(i>=f_begin-n) v = x->long_valid[i-(f_begin-n)];
    fmed[i] = v;
}
__global__ void fill_coord_kernel(Coord *dst, int from, int to, Coord v)
{
    const int i = from+blockIdx.x*blockDim.x+threadIdx.x;
    if(i<to) dst[i] = v;
}
__global__ void chain_skip_kernel(ChainCtx *x, int n) { chain_skip_clean_frames(x, n); x->next_frame += n; }
// The same with the count taken from device memory: frames [f, *first_unclean) were taken from the bulk pass (lazy verification).
__global__ void chain_skip_dev_kernel(ChainCtx *x, const int *first_unclean, int f) { const int n = *first_unclean-f; if(n>0) { chain_skip_clean_frames(x, n); x->next_frame += n; } }

// First frame in [from, n) whose clean flag is 0 (n if none) -> ctx->first_unclean.
__global__ void first_unclean_kernel(const u8 *clean, int from, int n, ChainCtx *x)
{
    __shared__ int s_min;
    if(threadIdx.x==0) s_min = n;
    __syncthreads();
    int m = n;
    for(int i=from+threadIdx.x;i<n;i+=blockDim.x) if(!(clean[2*i]&&clean[2*i+1])) { m = i; break; }      // both fields
    if(m<n) atomicMin(&s_min, m);
    __syncthreads();
    if(threadIdx.x==0) x->first_unclean = s_min;
}

// Rewrite black/white of the non-service records of frames [f0, f1) (the preset levels changed, nothing else did).
__global__ void patch_bw_kernel(sdv_line_rec *recs, size_t first, size_t count, u8 black, u8 white)
{
    size_t i = (size_t)blockIdx.x*blockDim.x+threadIdx.x;
    if(i<count)
    {
        sdv_line_rec *r = recs+first+i;
        if(r->service_type==SDV_SRV_NO) { r->black = black; r->white = white; }
    }
}

// ------------------------------------------------------------------------------------------------ deinterleave kernel
// Assembled line stream: index a -> record (or an empty line).  Two sources: a plain record array, or decoded frames
// laid out by the fixed geometry of sdv_stc007_frames_to_samples().
struct AsmMap
{
    const sdv_line_rec *recs;
    long long n_lines;          // plain array mode: number of lines; geometry mode: total assembled lines
    int geo;                    // 0 = plain array
    int lead_in, lpf, hf, H; long long n_fields;
    const sdv_line_rec *halo;   // geometry mode: the 112 line records that follow the last frame (next shard), or NULL
};
__device__ __forceinline__ const sdv_line_rec *asm_line(const AsmMap &m, long long a)
{
    if(!m.geo) return (a<m.n_lines) ? (m.recs+a) : (const sdv_line_rec *)0;
    a -= m.lead_in;
    if(a<0) return 0;
    long long fld = a/m.lpf; int j = (int)(a-fld*m.lpf);
    if(fld>=m.n_fields) return (m.halo&&(fld==m.n_fields)&&(j<112)&&(j<m.hf)) ? (m.halo+j) : (const sdv_line_rec *)0;
    if(j>=m.hf) return 0;
    return m.recs+((fld>>1)*m.H+(fld&1)*m.hf+j);
}

struct DeintParams
{
    AsmMap map; long long n_blocks;
    DeintCfg cfg;
    sdv_block_rec *blocks; i16 *samples; u8 *sflags;
    u32 *broken_bits;           // out: bit per block = BROKEN, not silent, not masked by a seam: may open a countdown window
    u8 *broken_sum;             // out: byte per 1024 blocks, set when one of their bits is
    // tile t of the launch covers blocks [tile_base + t*tile_stride, + tile_len) (0 / DEINT_TILE / DEINT_TILE = the whole stream);
    // other values: the blocks the fused bulk pass leaves over (stc007_bulk_kernel<true>), candidate bits set with atomics
    long long tile_base; int tile_stride, tile_len, n_tiles, atomic_bits;
};

// Samples, flags and the block record of one finished block.
__device__ __forceinline__ void block_store(const Block &blk, bool unsafe, long long b, sdv_block_rec *blocks, i16 *samples, u8 *sflags)
{
    if(samples||sflags)
    {
        i16 smp[6]; u8 fl[6];
        blk_output(&blk, smp, fl);
        u32 f03, f45;
        blk_output_flags(&blk, &f03, &f45);
        if(samples)
        {
            u32 *d = (u32 *)(samples+b*6);
            d[0] = (u32)(u16)smp[0]|((u32)(u16)smp[1]<<16); d[1] = (u32)(u16)smp[2]|((u32)(u16)smp[3]<<16); d[2] = (u32)(u16)smp[4]|((u32)(u16)smp[5]<<16);
        }
        if(sflags)
        {
            u16 *d = (u16 *)(sflags+b*6);
            d[0] = (u16)f03; d[1] = (u16)(f03>>16); d[2] = (u16)f45;
        }
    }
    if(blocks) blk_export(&blk, unsafe, blocks+b);
}

// One warp = one tile of DEINT_TILE consecutive data blocks: it stages the DEINT_TILE+112 line records the tile touches
// into its own piece of shared memory (every lane has ~8 independent 32-byte loads in flight), synchronises only
// with itself, and each lane then finishes 4 blocks.  No block-wide barrier: warps overlap each other's load latency.
enum { DEINT_WARPS = 8, DEINT_TILE = 128, DEINT_TLINES = DEINT_TILE+112, DEINT_THREADS = DEINT_WARPS*32, DEINT_CTA_BLOCKS = DEINT_WARPS*DEINT_TILE };

// PAIR: the standard setting with samples and flags only, an even first block and 8- / 4-byte aligned sample / flag buffers
// (deint_pair_applies): each lane finishes two adjacent blocks at once.
template<bool PAIR> __global__ void __launch_bounds__(DEINT_THREADS) stc007_deint_kernel(DeintParams p)
{
    __shared__ u16 s_wall[DEINT_WARPS][8][DEINT_TLINES];    // word-major: lane t reads s_w[k][t+16k], consecutive lanes consecutive addresses
    const int warp = threadIdx.x>>5, lane = threadIdx.x&31;
    u16 (*s_w)[DEINT_TLINES] = s_wall[warp];
    const long long tile = (long long)blockIdx.x*DEINT_WARPS+warp;
    if(tile>=p.n_tiles) return;
    const long long b0 = p.tile_base+tile*p.tile_stride;
    if(b0>=p.n_blocks) return;
    // position of assembled line b0 in the field grid (block counts are ints at the C ABI: 32-bit arithmetic is enough)
    int fld0 = 0, j0 = 0;
    const int n_fields = (int)p.map.n_fields, lpf = p.map.lpf, hf = p.map.hf;
    if(p.map.geo)
    {
        const int a0 = (int)b0-p.map.lead_in;
        const int q = (a0>=0) ? (a0/lpf) : -((-a0+lpf-1)/lpf);
        fld0 = q;
        j0 = a0-q*lpf;
    }
    // Geometry mode with the usual field length (>= the tile's 240 lines): the tile touches two fields at most; their
    // record pointers and line counts are uniform over the warp.
    const bool two_fields = p.map.geo&&(lpf>=DEINT_TLINES);
    const sdv_line_rec *fp[2] = { 0, 0 }; int fn[2] = { 0, 0 };
    if(two_fields)
    {
#pragma unroll
        for(int q=0;q<2;q++)
        {
            const int fld = fld0+q;
            if(fld<0) continue;
            if(fld<n_fields) { fp[q] = p.map.recs+((unsigned long long)(u32)(fld>>1)*(u32)p.map.H+(u32)((fld&1)*hf)); fn[q] = hf; }
            else if(p.map.halo&&(fld==n_fields)) { fp[q] = p.map.halo; fn[q] = (hf<112) ? hf : 112; }
        }
    }
    u32 okw[(DEINT_TLINES+31)/32];          // bit l of okw[it] = line 32*it+l of the tile gives trusted words (same in every lane)
    auto line_ptr = [&](int ln) -> const sdv_line_rec *
    {
        if(ln>=DEINT_TLINES) return 0;
        if(!p.map.geo) return (b0+ln<p.map.n_lines) ? (p.map.recs+b0+ln) : (const sdv_line_rec *)0;
        if(two_fields)
        {
            int j = j0+ln;
            const int q = (j>=lpf) ? 1 : 0;
            j -= q ? lpf : 0;
            return (j<(q ? fn[1] : fn[0])) ? ((q ? fp[1] : fp[0])+j) : (const sdv_line_rec *)0;
        }
        int j = j0+ln, fld = fld0;
        while(j>=lpf) { j -= lpf; fld++; }
        if((fld<0)||(j>=hf)) return 0;
        if(fld>=n_fields) return (p.map.halo&&(fld==n_fields)&&(j<112)) ? (p.map.halo+j) : (const sdv_line_rec *)0;
        return p.map.recs+((unsigned long long)(u32)(fld>>1)*(u32)p.map.H+(u32)((fld&1)*hf+j));
    };
    // one lane per line, the 32-byte record as two 16-byte loads; DEINT_GROUP lines' loads are issued before the first
    // is used (the wait for a record was the largest single stall of this kernel)
    enum { DEINT_GROUP = 4 };
#pragma unroll
    for(int g=0;g<(DEINT_TLINES+31)/32;g+=DEINT_GROUP)
    {
        const sdv_line_rec *r[DEINT_GROUP];
        uint4 wv[DEINT_GROUP], tv[DEINT_GROUP];
#pragma unroll
        for(int i=0;i<DEINT_GROUP;i++) r[i] = line_ptr(lane+32*(g+i));
#pragma unroll
        for(int i=0;i<DEINT_GROUP;i++)
        {
            wv[i] = make_uint4(0, 0, 0, 0); tv[i] = make_uint4(0, 0, 0, 0);
            if(r[i]) { wv[i] = __ldg((const uint4 *)r[i]); tv[i] = __ldg((const uint4 *)r[i]+1); }    // words | CRCC|flags, ref.., data_start|data_stop, shift|service|marks
        }
#pragma unroll
        for(int i=0;i<DEINT_GROUP;i++)
        {
            const int ln = lane+32*(g+i);
            const uint4 t = tv[i];
            const u32 fl = t.x>>16;
            bool ok = false;
            if(r[i]&&(((t.w>>8)&0xFFu)==SDV_SRV_NO))
            {
                if(!p.cfg.ignore_crc) ok = (fl&SDV_LF_CRC_OK)!=0;
                else { Coord cc; cc.start = (i16)(t.z&0xFFFFu); cc.stop = (i16)(t.z>>16); ok = coord_valid(cc)&&((fl&SDV_LF_BW_SET)!=0); }
            }
            if(ln<DEINT_TLINES)
            {
                s_w[0][ln] = (u16)wv[i].x; s_w[1][ln] = (u16)(wv[i].x>>16); s_w[2][ln] = (u16)wv[i].y; s_w[3][ln] = (u16)(wv[i].y>>16);
                s_w[4][ln] = (u16)wv[i].z; s_w[5][ln] = (u16)(wv[i].z>>16); s_w[6][ln] = (u16)wv[i].w; s_w[7][ln] = (u16)(wv[i].w>>16);
            }
            okw[g+i] = __ballot_sync(0xFFFFFFFFu, ok);
        }
    }
    __syncwarp();
    // The standard setting with samples and flags only: each lane takes blocks s and s+1 (s even) at once, as packed word pairs
    // (stc007_deint.cuh, deint_pair_std14) -- word k of lines s+16k and s+1+16k is one 32-bit shared load, their trusted bits
    // one 2-bit field of the ballot windows -- and stores 24 bytes of samples and 12 of flags.  Pairs it does not cover, and a
    // block whose partner lies past the tile or the stream, go through deint_block_std14() one by one.
    if constexpr(PAIR)
    {
        const int n_here = (int)(((long long)p.tile_len<p.n_blocks-b0) ? (long long)p.tile_len : (p.n_blocks-b0));
        u32 lw[(DEINT_TLINES+31)/32-1];     // the window words from this half-warp's first line on: lanes 16..31 start 32 lines later
#pragma unroll
        for(int i=0;i<(DEINT_TLINES+31)/32-1;i++) lw[i] = (lane<16) ? okw[i] : okw[i+1];
        // Both pairs of the lane first, as two independent branch-free chains; then their stores, or the one-block path
        u32 d[DEINT_TILE/64][6], f[DEINT_TILE/64][3], bnp[DEINT_TILE/64], okf[DEINT_TILE/64][4];
        bool cov[DEINT_TILE/64];
#pragma unroll
        for(int jt=0;jt<DEINT_TILE/64;jt++)
        {
            const int s = 2*lane+64*jt;
            u32 w[8];       // (lines s+16k, s+1+16k < DEINT_TLINES: always inside the staged tile)
#pragma unroll
            for(int k=0;k<8;k++) w[k] = *(const u32 *)&s_w[k][s+16*k];
            // bits 0 / 1: line s+32m / s+1+32m (word 2m of blocks s / s+1); bits 16 / 17: 16 lines on (word 2m+1)
#pragma unroll
            for(int m=0;m<4;m++) okf[jt][m] = __funnelshift_r(lw[2*jt+m], lw[2*jt+m+1], 2*lane);
            BlockPair bp;
            cov[jt] = deint_pair_std14(w, okf[jt], &bp);
            pair_samples(&bp, d[jt]);
            pair_flags(&bp, f[jt]);
            bnp[jt] = pair_broken_ns(&bp);
        }
#pragma unroll
        for(int jt=0;jt<DEINT_TILE/64;jt++)
        {
            const int s = 2*lane+64*jt;
            const long long b = b0+s;
            u32 bns = 0;    // bit h: block s+h is BROKEN and not silent
            if(cov[jt]&&(s+1<n_here))
            {
                uint2 *sd = (uint2 *)(p.samples+b*6);
                sd[0] = make_uint2(d[jt][0], d[jt][1]); sd[1] = make_uint2(d[jt][2], d[jt][3]); sd[2] = make_uint2(d[jt][4], d[jt][5]);
                u32 *fd = (u32 *)(p.sflags+b*6);
                fd[0] = f[jt][0]; fd[1] = f[jt][1]; fd[2] = f[jt][2];
                bns = bnp[jt];
            }
            else
            {
                for(int h=0;h<2;h++)
                {
                    if(s+h>=n_here) break;
                    BlockIn in; in.ok = 0;
#pragma unroll
                    for(int k=0;k<8;k++)
                    {
                        const int ln = s+h+16*k;
                        in.w[k] = s_w[k][ln]; in.sw[k] = s_w[7][ln];
                        in.ok |= (u8)(((okf[jt][k>>1]>>(16*(k&1)+h))&1u)<<k);
                    }
                    Block blk;
                    deint_block_std14(&blk, &in);
                    blk.m2 = 0;
                    if((blk.audio_state==SDV_AUD_BROKEN)&&!blk_silent(&blk)) bns |= 1u<<h;
                    block_store(blk, false, b+h, p.blocks, p.samples, p.sflags);
                }
            }
            if(p.atomic_bits)
            {
                if(p.broken_bits)
                    for(int h=0;h<2;h++)
                        if((bns>>h)&1u) { atomicOr(&p.broken_bits[(b+h)>>5], 1u<<(u32)((b+h)&31)); p.broken_sum[(b+h)>>10] = 1; }
            }
            else
            {   // blocks 64jt..+31 are lanes 0..15, the next 32 lanes 16..31: lanes 0 and 16 write the two words
                const u32 v = bns<<((2*lane)&31);
                const u32 bal0 = __reduce_or_sync(0xFFFFFFFFu, (lane<16) ? v : 0u), bal1 = __reduce_or_sync(0xFFFFFFFFu, (lane<16) ? 0u : v);
                const u32 bal = (lane<16) ? bal0 : bal1;
                if(((lane&15)==0)&&(b<p.n_blocks))
                {
                    if(p.broken_bits) p.broken_bits[b>>5] = bal;
                    if(bal&&p.broken_sum) p.broken_sum[b>>10] = 1;
                }
            }
        }
        return;
    }
    for(int jt=0;jt<DEINT_TILE/32;jt++)
    {
        const int s = lane+32*jt;
        const long long b = b0+s;
        bool broken_ns = false;
        if((b<p.n_blocks)&&(s<p.tile_len))
        {
            BlockIn in; in.ok = 0;
#pragma unroll
            for(int k=0;k<8;k++)
            {
                const int ln = s+16*k;
                in.w[k] = s_w[k][ln]; in.sw[k] = s_w[7][ln];
                // line ln = 32*jt+16k+lane = bit (16*(k&1)+lane) of the 64-bit window okw[(k>>1)+1]:okw[k>>1] (okw is rotated by jt)
                const u32 win = (k&1) ? __funnelshift_r(okw[k>>1], okw[(k>>1)+1], 16) : okw[k>>1];
                in.ok |= (u8)(((win>>lane)&1u)<<k);
            }
            Block blk;
            deint_dispatch(&blk, &in, p.cfg);
            broken_ns = (blk.audio_state==SDV_AUD_BROKEN)&&!blk_silent(&blk);
            block_store(blk, false, b, p.blocks, p.samples, p.sflags);
        }
        const u32 bal = __ballot_sync(0xFFFFFFFFu, broken_ns);
        if(p.atomic_bits)
        {
            if(broken_ns&&p.broken_bits) { atomicOr(&p.broken_bits[b>>5], 1u<<(u32)(b&31)); p.broken_sum[b>>10] = 1; }
        }
        else if((lane==0)&&(b<p.n_blocks))
        {
            if(p.broken_bits) p.broken_bits[b>>5] = bal;
            if(bal&&p.broken_sum) p.broken_sum[b>>10] = 1;
        }
#pragma unroll
        for(int i=0;i+1<(DEINT_TLINES+31)/32;i++) okw[i] = okw[i+1];    // next 32 blocks: the window moves on by one word
    }
}

// The same pass over the stream of a StitchMap (frames stacked by the reference's own alignment decisions): one thread
// per data block, lines gathered through the frame descriptors; blocks across an untrusted seam are marked unsafe here.
struct StitchDeintParams
{
    StitchMap map; long long n_blocks;
    DeintCfg cfg;
    sdv_block_rec *blocks; i16 *samples; u8 *sflags;
    u32 *broken_bits; u8 *broken_sum;
};
__global__ void __launch_bounds__(256) stc007_stitch_deint_kernel(StitchDeintParams p)
{
    const long long b = (long long)blockIdx.x*256+threadIdx.x;
    bool broken_ns = false;
    if(b<p.n_blocks)
    {
        int hint = (int)((b-p.map.n_carry-p.map.lead)/p.map.frame_len);
        BlockIn in;
        DeintCfg cfg = p.cfg;
        const bool masked = stitch_block_in(p.map, b, p.cfg.ignore_crc!=0, &in, &hint, &cfg.res_mode);
        Block blk;
        deint_dispatch(&blk, &in, cfg);
        const bool silent = blk_silent(&blk);
        bool unsafe = false;
        if(masked&&!silent) { unsafe = (blk.audio_state!=SDV_AUD_BROKEN); blk_mark_unsafe(&blk); }
        broken_ns = (blk.audio_state==SDV_AUD_BROKEN)&&(!silent)&&(!masked);
        block_store(blk, unsafe, b, p.blocks, p.samples, p.sflags);
    }
    const u32 bal = __ballot_sync(0xFFFFFFFFu, broken_ns);
    if(((threadIdx.x&31)==0)&&(b<p.n_blocks))
    {
        p.broken_bits[b>>5] = bal;
        if(bal) p.broken_sum[b>>10] = 1;
    }
}

// ------------------------------------------------------------------------------------------------ broken-block countdown
// STC007DataStitcher::performDeinterleave (stc007datastitcher.cpp:6778-6800,6859-6862): a BROKEN block (not silent, not
// already masked by a seam) met with the countdown at 0 opens a window of [dur] blocks in which every block that is not
// silent and not seam-masked is marked unsafe.  The windows are a sequential function of the sparse list of such blocks:
// one thread block walks it (whole 1024-block groups without a candidate are skipped by their summary byte) and writes
// the window list; stc007_window_kernel then redoes just the blocks inside windows with the mark applied.
// state[0] in: countdown left over from the blocks before this stream (0 at a file start); state[1] out: the countdown
// after the last block; state[2] out: number of windows; state[3] out: a candidate lies within the first [dur] blocks
// (only then can state[0] change anything but the marks of the first blocks).
struct WindowList { long long *start; int *len; int cap; int *state; };
__global__ void __launch_bounds__(1024) broken_window_kernel(const u32 *broken_bits, const u8 *broken_sum, long long n_blocks, int dur, int countdown_in, WindowList wl)
{
    if(threadIdx.x==0) wl.state[0] = countdown_in;
    __shared__ int s_groups[1024];
    __shared__ int s_n;
    const long long n_groups = (n_blocks+1023)>>10, n_words = (n_blocks+31)>>5;
    long long open_until = countdown_in;
    int n_win = 0, depends = 0;
    {   // a tape without a single candidate (every clean tape): one pass over the summary bytes instead of the walk
        int any = 0;
        for(long long g=threadIdx.x;g<n_groups;g+=blockDim.x) any |= broken_sum[g];
        if(!__syncthreads_or(any))
        {
            if(threadIdx.x==0)
            {
                const int w0 = (open_until>0) ? 1 : 0;
                if(w0&&(wl.cap>0)) { wl.start[0] = 0; wl.len[0] = (int)((open_until<n_blocks) ? open_until : n_blocks); }
                wl.state[1] = (int)((open_until>n_blocks) ? (open_until-n_blocks) : 0);
                wl.state[2] = (w0<wl.cap) ? w0 : wl.cap;
                wl.state[3] = 0;
            }
            return;
        }
    }
    if((threadIdx.x==0)&&(open_until>0)&&(n_win<wl.cap)) { wl.start[0] = 0; wl.len[0] = (int)((open_until<n_blocks) ? open_until : n_blocks); }
    if(open_until>0) n_win = 1;
    for(long long g0=0;g0<n_groups;g0+=1024)
    {
        // groups with a candidate, in order
        if(threadIdx.x==0) s_n = 0;
        __syncthreads();
        const long long g = g0+threadIdx.x;
        const bool hit = (g<n_groups)&&(broken_sum[g]!=0);
        const u32 bal = __ballot_sync(0xFFFFFFFFu, hit);
        __shared__ int s_wcnt[32];
        if((threadIdx.x&31)==0) s_wcnt[threadIdx.x>>5] = __popc(bal);
        __syncthreads();
        if(hit)
        {
            int pos = __popc(bal&((1u<<(threadIdx.x&31))-1u));
            for(int w=0;w<(int)(threadIdx.x>>5);w++) pos += s_wcnt[w];
            s_groups[pos] = threadIdx.x;
        }
        if(threadIdx.x==0) { int t = 0; for(int w=0;w<32;w++) t += s_wcnt[w]; s_n = t; }
        __syncthreads();
        if(threadIdx.x<32)
        {
            const int lane = threadIdx.x;
            for(int i=0;i<s_n;i++)
            {
                const long long wi = ((g0+s_groups[i])<<5)+lane;
                u32 v = (wi<n_words) ? broken_bits[wi] : 0u;
                u32 nz = __ballot_sync(0xFFFFFFFFu, v!=0);
                while(nz)
                {
                    const int src = __ffs(nz)-1; nz &= nz-1;
                    u32 bits = __shfl_sync(0xFFFFFFFFu, v, src);
                    while(bits)
                    {
                        const int bit = __ffs(bits)-1; bits &= bits-1;
                        const long long blk = ((((g0+s_groups[i])<<5)+src)<<5)+bit;
                        if(blk<dur) depends = 1;
                        if(blk>=open_until)
                        {
                            open_until = blk+dur;
                            if((lane==0)&&(n_win<wl.cap)) { wl.start[n_win] = blk; wl.len[n_win] = (int)((blk+dur<=n_blocks) ? dur : (n_blocks-blk)); }
                            n_win++;
                        }
                    }
                }
            }
        }
        __syncthreads();
    }
    if(threadIdx.x==0)
    {
        wl.state[1] = (int)((open_until>n_blocks) ? (open_until-n_blocks) : 0);
        wl.state[2] = (n_win<wl.cap) ? n_win : wl.cap;
        wl.state[3] = depends;
    }
}

// Blocks inside countdown windows once more, with the mark.  One thread block per window (grid-stride over the list).
struct WindowParams
{
    int stitched; AsmMap amap; StitchMap smap; long long n_blocks;
    int from_records;           // CWD: the blocks are not recomputed from the line records (CWD patched the lines) but taken from [blocks]
    DeintCfg cfg;
    sdv_block_rec *blocks; i16 *samples; u8 *sflags;
    WindowList wl;
};
__global__ void __launch_bounds__(128) stc007_window_kernel(WindowParams p)
{
    const int n_win = p.wl.state[2];
    for(int w=blockIdx.x;w<n_win;w+=gridDim.x)
    {
        const long long b0 = p.wl.start[w]; const int len = p.wl.len[w];
        for(int q=threadIdx.x;q<len;q+=blockDim.x)
        {
            const long long b = b0+q;
            if(b>=p.n_blocks) break;
            if(p.from_records)
            {
                const sdv_block_rec r = p.blocks[b];
                if(r.flags&(SDV_BF_SILENT|SDV_BF_UNSAFE)) continue;     // silent blocks are left alone, seam-masked ones carry their mark already
                Block blk;
                for(int k=0;k<8;k++) blk.words[k] = r.words[k];
                blk.line_crc = r.line_crc; blk.word_valid = r.word_valid; blk.resolution = r.resolution; blk.audio_state = r.audio_state; blk.m2 = p.cfg.m2;
                const bool unsafe = (blk.audio_state!=SDV_AUD_BROKEN);
                blk_mark_unsafe(&blk);
                block_store(blk, unsafe, b, p.blocks, p.samples, p.sflags);
                continue;
            }
            BlockIn in; bool masked = false;
            DeintCfg cfg = p.cfg;
            if(p.stitched)
            {
                int hint = (int)((b-p.smap.n_carry-p.smap.lead)/p.smap.frame_len);
                masked = stitch_block_in(p.smap, b, p.cfg.ignore_crc!=0, &in, &hint, &cfg.res_mode);
            }
            else
            {
                in.ok = 0;
#pragma unroll
                for(int k=0;k<8;k++)
                {
                    const sdv_line_rec *r = asm_line(p.amap, b+16*k);
                    u16 wd = 0, sw = 0; bool ok = false;
                    if(r) { wd = r->words[k]; sw = r->words[7]; ok = line_rec_ok(r, p.cfg.ignore_crc!=0); }
                    in.w[k] = wd; in.sw[k] = sw;
                    if(ok) in.ok |= (u8)(1u<<k);
                }
            }
            Block blk;
            deint_dispatch(&blk, &in, cfg);
            if(masked||blk_silent(&blk)) continue;      // silent blocks are left alone, seam-masked ones carry their mark already
            const bool unsafe = (blk.audio_state!=SDV_AUD_BROKEN);
            blk_mark_unsafe(&blk);
            block_store(blk, unsafe, b, p.blocks, p.samples, p.sflags);
        }
    }
}

// ------------------------------------------------------------------------------------------------ seam sweep
// STC007DataStitcher::tryPadding (stc007datastitcher.cpp:1417-1740) for a list of (seam, padding range) tasks: one thread
// block per (task, padding) candidate, one thread per data block of the seam queue (tail of field 1, [padding] empty
// lines, head of field 2 -- an index map, never materialised), 128 blocks at a time, the reference's burst counters
// replayed by thread 0 over the flags (stc007_stitch.cuh).
enum { SEAM_THREADS = 128 };
struct SeamParams
{
    const sdv_line_rec *recs; const SeamTask *tasks; int n_tasks;
    DeintCfg cfg; int lim14, lim16;
    sdv_stitch_stats *out;
};
__global__ void __launch_bounds__(SEAM_THREADS) stc007_seam_kernel(SeamParams p)
{
    __shared__ u8 s_flags[SEAM_THREADS];
    const SeamTask t = p.tasks[blockIdx.x];
    if((int)blockIdx.y>=(int)t.n_pad) return;
    const int pad = t.pad0+blockIdx.y;
    const SeamGeom g = seam_geom(t.f1.size, t.f2.size, pad);
    const int lim = p.cfg.q_corr ? p.lim14 : p.lim16;
    DeintCfg cfg = p.cfg; cfg.res_mode = seam_queue_res_mode(t, g, p.cfg.res_mode);
    SeamCount cnt; seam_count_init(&cnt);
    for(int base=0;base<g.nblk;base+=SEAM_THREADS)
    {
        const int s = base+threadIdx.x;
        s_flags[threadIdx.x] = (s<g.nblk) ? seam_block_flags(p.recs, t, g, s, cfg) : (u8)0;
        __syncthreads();
        if(threadIdx.x==0) { const int m = (g.nblk-base<SEAM_THREADS) ? (g.nblk-base) : SEAM_THREADS; for(int i=0;i<m;i++) seam_count_step(&cnt, s_flags[i], lim); }
        __syncthreads();
    }
    if(threadIdx.x==0) p.out[t.out+blockIdx.y] = seam_count_finish(&cnt, g, lim);
}
// sdv_seam (the C ABI's plain field ranges) -> tasks sweeping paddings 0..n_pad-1
__global__ void seam_tasks_kernel(const sdv_seam *seams, int n, int n_pad, SeamTask *tasks)
{
    const int i = blockIdx.x*blockDim.x+threadIdx.x;
    if(i>=n) return;
    SeamTask t;
    t.f1.first = seams[i].f1_first; t.f1.size = (u16)seams[i].f1_size; t.f1.hole = ST_NO_HOLE;
    t.f2.first = seams[i].f2_first; t.f2.size = (u16)seams[i].f2_size; t.f2.hole = ST_NO_HOLE;
    t.pad0 = 0; t.n_pad = (u16)n_pad; t.out = (u32)i*(u32)n_pad; t.res1 = t.res2 = RES_ANY; t.pad_[0] = t.pad_[1] = 0;
    tasks[i] = t;
}

// ------------------------------------------------------------------------------------------------ frame trim
// findFramesTrim + splitFramesToFields for every frame: one thread block per frame (stc007_stitch.cuh).
__global__ void __launch_bounds__(128) stc007_trim_kernel(const sdv_line_rec *recs, int n_frames, int H, FrameTrim *out)
{
    __shared__ int scr[8];
    const Cta c = { (int)threadIdx.x, (int)blockDim.x };
    const int f = blockIdx.x, hf = H/2;
    trim_field_cta(c, recs+(size_t)f*H, hf, 0, scr, &out[f].odd);
    trim_field_cta(c, recs+(size_t)f*H+hf, hf, 1, scr, &out[f].even);
}


// ------------------------------------------------------------------------------------------------ audio resolution per field
// STC007DataStitcher::getFieldResolution (stc007datastitcher.cpp:996-1195) for both fields of every frame: one thread block
// per field, one thread per data block inside the trimmed field (14-bit and 16-bit try), the reference's two saturating
// counters replayed in block order by thread 0.  out[2*f + even] = ST_RES_*.
__global__ void __launch_bounds__(128) stc007_fieldres_kernel(const sdv_line_rec *recs, const FrameTrim *trims, int H, u8 *out)
{
    __shared__ u8 s_flags[128];
    const int f = blockIdx.x>>1, even = blockIdx.x&1;
    const FieldTrim t = even ? trims[f].even : trims[f].odd;
    SeamField fld; fld.first = (u32)((size_t)f*H+(even ? H/2 : 0)+t.first); fld.size = t.data_lines; fld.hole = t.hole;
    const int n = (t.data_lines>112) ? (t.data_lines-112) : 0;
    int c14 = 0, c16 = 0;
    for(int base=0;base<n;base+=128)
    {
        const int i = base+threadIdx.x;
        s_flags[threadIdx.x] = (i<n) ? field_res_flags(recs, fld, i, false) : (u8)0;
        __syncthreads();
        if(threadIdx.x==0) { const int m = (n-base<128) ? (n-base) : 128; for(int k=0;k<m;k++) field_res_step(&c14, &c16, s_flags[k]); }
        __syncthreads();
    }
    if(threadIdx.x==0) out[blockIdx.x] = n ? field_res_decide(c14, c16) : (u8)ST_RES_UNKNOWN;
}

// ------------------------------------------------------------------------------------------------ CWD
// Frames that hold a line CWD may write into (out[f] != 0): one thread block per frame.
__global__ void __launch_bounds__(128) stc007_cwd_scan_kernel(const sdv_line_rec *recs, int H, u8 *out)
{
    const sdv_line_rec *r = recs+(size_t)blockIdx.x*H;
    int any = 0;
    for(int j=threadIdx.x;j<H;j+=blockDim.x) if(rec_cwd_patchable(r+j)) any = 1;
    any = __syncthreads_or(any);
    if(threadIdx.x==0) out[blockIdx.x] = any ? 1 : 0;
}
// One chain of consecutive frames per thread block (stc007_cwd.cuh).
__global__ void __launch_bounds__(CWD_THREADS) stc007_cwd_chain_kernel(CwdParams p)
{
    __shared__ CwdShared sh;
    const Cta c = { (int)threadIdx.x, (int)blockDim.x };
    cwd_chain_cta(c, p, blockIdx.x, &sh);
}
// Speculative walk: does frame S (dirty, not the first of its chain) hold the lines its predecessor left?  ok[S] = 1 / 0.
__global__ void __launch_bounds__(128) cwd_verify_kernel(const int *steps, int n, const CwdLine *step_out, const CwdLine *step_used, const u16 *step_n, u8 *ok)
{
    const int S = steps[blockIdx.x];
    const int n_used = step_n[2*S], n_out = step_n[2*(S-1)+1];
    int bad = (n_used!=n_out) ? 1 : 0;
    if(!bad)
    {
        const u32 *a = (const u32 *)(step_used+(size_t)S*112), *b = (const u32 *)(step_out+(size_t)(S-1)*112);
        for(int i=threadIdx.x;i<n_used*(int)(sizeof(CwdLine)/4);i+=blockDim.x) if(a[i]!=b[i]) bad = 1;
    }
    bad = __syncthreads_or(bad);
    if(threadIdx.x==0) ok[blockIdx.x] = bad ? 0 : 1;
    (void)n;
}

}   // namespace sdv

// ================================================================================================ C ABI
using namespace sdv;

struct sdv_handle
{
    int device, num_sms;
    ChainCtx *ctx;              // device
    u8 *clean; size_t clean_cap;
    u32 *bits; size_t bits_cap; // candidate bits, their 1024-block summary, the countdown window list (run_deint)
    int *win_state;             // device: countdown in / out, number of windows, dependence flag (broken_window_kernel)
    int *win_state_host;        // pinned copy
    // STC-007 stitcher (sdv_stc007_stitch_frames)
    FrameTrim *trim_dev; size_t trim_cap;
    FrameAsm *fa_dev; size_t fa_cap;
    SeamTask *task_dev; size_t task_cap;
    sdv_stitch_stats *sstat_dev; size_t sstat_cap;
    sdv_line_rec *carry_dev[2]; i32 *carry_meta_dev[2]; int carry_cur, carry_valid;   // the 112 lines a call leaves in the queue for the next
    StitchCarry st_carry; int st_frame_base; int st_countdown; ResChain st_res;
    int st_flags;               // SB_FLAG_* of the call that left the open file (what a saved state records)
    int st_loaded;              // the open file came from sdv_stc007_stitch_state_load: the next call must match st_flags
    u8 *fres_dev; size_t fres_cap;  // detected resolution per field + the four modes per frame
    // CWD
    u8 *cwd_scan_dev; size_t cwd_scan_cap; u8 *cwd_plan_dev; size_t cwd_plan_cap; int *cwd_status;
    CwdLine *cwd_carry[2]; int cwd_carry_valid;     // the patched lines a call leaves in the queue (beside carry_dev, same slot index)
    sdv_block_rec *blk_scratch; size_t blk_scratch_cap;
    u8 *cwd_spec_dev; size_t cwd_spec_cap;      // speculative CWD walk: lines every frame took / left
    FineSet fine;               // Binarizer fine settings of this handle (sdv_bin_set_fine_settings)
    // fused deinterleave (sdv_stc007_fuse_next_decode): what the next decode call shall also produce / what the last one did
    struct { int armed; sdv_deint_config cfg; sdv_stc007_geometry geo; int16_t *samples; uint8_t *sflags; } fuse_arm;
    struct { int valid, n_frames, H, f_from, lead_in, lpf, dur; int16_t *samples; uint8_t *sflags; const sdv_line_rec *recs; } fuse_done;
    // lazy verification of the warm-start pass (sdv_bin_config.reserved[2] bit 1, sdv_bin_decode_verify)
    int lazy_pending; cudaEvent_t ev_lazy;
    sdv_bin_config lazy_cfg; const uint8_t *lazy_luma; int lazy_n, lazy_H, lazy_W, lazy_stride; sdv_line_rec *lazy_recs; sdv_line_aux *lazy_aux; void *lazy_stream;
    X0PadChain x0_pads; int x0_pads_open;        // PCM-16x0 SI padding history (sdv_pcm16x0_frames_to_samples_auto)
    X0EIScan *x0_scan_ei; size_t x0_scan_ei_cap;
    X0PadScan *x0_scan; size_t x0_scan_cap; X0FieldGeo *x0_geo; size_t x0_geo_cap; u8 *x0_mask; size_t x0_mask_cap;
    u8 *pad_dev; size_t pad_cap; // seams + statistics of sdv_stc007_find_padding
    ChainHdr *hdr_host;         // pinned copy of the first bytes of ctx
    ChainCtx *seg_ctx; size_t seg_cap;      // one context per segment (segment mode) / per piece (relay mode: end states)
    ChainCtx *start_ctx; size_t start_cap;  // relay mode: state at the head of every piece
    Coord *fmed; size_t fmed_cap;           // per-frame coordinate medians
    ChainSnap *snaps; size_t snaps_cap;     // relay mode: chain state at the head of every frame
    sdv_line_rec *warm_scratch; size_t warm_cap;
    u8 *relay_ok; size_t relay_ok_cap; u8 *relay_ok_host; size_t relay_ok_host_cap;
    int warm_valid, warm_H, warm_W, warm_mode; BinState warm_bin;      // presets the last decode ended with
    int chain_open, chain_H, chain_W, chain_mode;                      // ctx holds the chain state at the end of the last STC-007 decode
    int *spec_fu, *fu_host;                 // first unclean frame of the speculative bulk launch (device / pinned host)
    cudaEvent_t ev_sync[2];
    sdv_first_frame_fn first_frame_fn; void *first_frame_user; int first_frame_called;
    sdv_bin_stats stats;
    // staging for the host-buffer entry point
    u8 *luma_dev; size_t luma_cap;
    sdv_line_rec *recs_dev; size_t recs_cap;
    i16 *smp_dev; u8 *sfl_dev; size_t smp_cap;
    cudaStream_t stream, copy_stream;
    cudaEvent_t ev[4];          // timing: bulk kernel begin/end, deinterleave kernel begin/end (last launch of each)
    int ev_set[2]; uint64_t ev_units[2];
    double acc_ms[2]; uint64_t acc_units[2]; uint32_t acc_n[2]; uint32_t acc_launches;
    // PCM-1 line decode
    P1Preset *p1_scan; size_t p1_scan_cap;        // four prescan results per frame
    P1Preset *p1_presets; size_t p1_presets_cap;  // per-frame presets
    u8 *p1_clean; size_t p1_clean_cap;
    u32 *p1_bw; size_t p1_bw_cap;
    P1ChainCtx *p1_ctx;
    X0ChainCtx *x0_ctx;
    int pcm_open, pcm_type, pcm_H, pcm_W, pcm_mode;    // p1_ctx / x0_ctx hold the chain state at the end of the last PCM-1 / PCM-16x0 decode
    u8 *x0_votes; int x0_votes_cur, x0_votes_open;     // control-bit votes of the last X0_CTRL_HISTORY frames of the PCM-16x0 stitch calls (two buffers)
    unsigned long long *p1_stats_dev, *p1_stats_host;
    sdv_pcm1_subline *p1_sub; size_t p1_sub_cap;  // assembled fields (sdv_pcm1_frames_to_samples)
    char err[256];
};

static int fail(sdv_handle *h, int code, const char *what, cudaError_t e)
{
    if(h) snprintf(h->err, sizeof(h->err), "%s: %s", what, (e==cudaSuccess) ? "invalid argument" : cudaGetErrorString(e));
    return code;
}
#define CK(call) do { cudaError_t e_ = (call); if(e_!=cudaSuccess) return fail(h, SDV_ERR_CUDA, #call, e_); } while(0)

static void crc_tables(u16 *bit, u16 *zero)
{
    // message = 8 x 14 bits, MSB first; contribution of message bit i = CRC (init 0) of the unit message e_i
    for(int i=0;i<112;i++)
    {
        u16 w[8] = {0};
        w[i/14] = (u16)(1u<<(13-(i%14)));
        u16 c = 0; for(int k=0;k<8;k++) c = crc16_update(c, w[k], 14);
        bit[i] = c;
    }
    u16 z[8] = {0};
    *zero = crc_stc007(z);
}

extern "C" {

int sdv_version(void) { return 100; }

const char *sdv_last_error(sdv_handle *h) { return h ? h->err : "null handle"; }

int sdv_create(sdv_handle **out, int cuda_device)
{
    if(!out) return SDV_ERR_ARG;
    *out = NULL;
    int n = 0;
    if((cudaGetDeviceCount(&n)!=cudaSuccess)||(n<=0)||(cuda_device<0)||(cuda_device>=n)) return SDV_ERR_CUDA;   // no CPU fallback
    sdv_handle *h = new (std::nothrow) sdv_handle();
    if(!h) return SDV_ERR_NOMEM;
    memset(h, 0, sizeof(*h));
    { const FineSet d = SDV_FINE_DEFAULTS; h->fine = d; }
    h->device = cuda_device;
    cudaError_t e = cudaSetDevice(cuda_device);
    if(e==cudaSuccess) e = cudaMalloc(&h->ctx, sizeof(ChainCtx));
    if(e==cudaSuccess) e = cudaMallocHost(&h->hdr_host, sizeof(ChainHdr));
    if(e==cudaSuccess) e = cudaMallocHost(&h->fu_host, sizeof(int));
    if(e==cudaSuccess) e = cudaMalloc(&h->spec_fu, sizeof(int));
    if(e==cudaSuccess) e = cudaMalloc(&h->win_state, 4*sizeof(int));
    if(e==cudaSuccess) e = cudaMemset(h->win_state, 0, 4*sizeof(int));
    if(e==cudaSuccess) e = cudaMallocHost(&h->win_state_host, 4*sizeof(int));
    for(int i=0;(i<2)&&(e==cudaSuccess);i++)
    {
        e = cudaMalloc(&h->carry_dev[i], ST_TAIL*sizeof(sdv_line_rec));
        if(e==cudaSuccess) e = cudaMalloc(&h->carry_meta_dev[i], 2*ST_TAIL*sizeof(i32));
        if(e==cudaSuccess) e = cudaMalloc(&h->cwd_carry[i], ST_TAIL*sizeof(CwdLine));
    }
    if(e==cudaSuccess) e = cudaMalloc(&h->cwd_status, sizeof(int));
    if(e==cudaSuccess) e = cudaMemset(h->cwd_status, 0, sizeof(int));
    for(int i=0;(i<2)&&(e==cudaSuccess);i++) e = cudaEventCreateWithFlags(&h->ev_sync[i], cudaEventDisableTiming);
    if(e==cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_lazy, cudaEventDisableTiming);
    if(e==cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if(e==cudaSuccess) e = cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
    for(int i=0;(i<4)&&(e==cudaSuccess);i++) e = cudaEventCreate(&h->ev[i]);
    if(e==cudaSuccess)
    {
        u16 bit[112], zero;
        crc_tables(bit, &zero);
        e = cudaMemcpyToSymbol(c_crc_bit, bit, sizeof(bit));
        if(e==cudaSuccess) e = cudaMemcpyToSymbol(c_crc_zero, &zero, sizeof(zero));
    }
    if(e==cudaSuccess)
    {
        u16 tab[3*256];
        for(int i=0;i<256;i++)
        {
            tab[i] = crc16_update(0, (u16)i, 8);
            u16 lo = (u16)i, hi = (u16)(i<<8);                  // CRC state advanced over 7 zero bytes (linear in the state)
            for(int k=0;k<7;k++) { lo = crc16_update(lo, 0, 8); hi = crc16_update(hi, 0, 8); }
            tab[256+i] = lo; tab[512+i] = hi;
        }
        e = cudaMemcpyToSymbol(c_crc8, tab, sizeof(tab));
    }
    if(e==cudaSuccess) e = cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, cuda_device);
    if(e==cudaSuccess) e = cudaFuncSetAttribute(stc007_bulk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227*1024);
    if(e==cudaSuccess) e = cudaFuncSetAttribute(stc007_bulk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227*1024);
    if(e==cudaSuccess) e = cudaFuncSetAttribute(pcm1_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(P1ChainCtx));
    if(e==cudaSuccess) e = cudaFuncSetAttribute(pcm16x0_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(X0ChainCtx));
    if(e==cudaSuccess) e = cudaFuncSetAttribute(pcm1_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227*1024);
    if(e==cudaSuccess) e = cudaMalloc(&h->p1_ctx, sizeof(P1ChainCtx));
    if(e==cudaSuccess) e = cudaMalloc(&h->x0_ctx, sizeof(X0ChainCtx));
    if(e==cudaSuccess) e = cudaMalloc(&h->x0_votes, 2*X0_CTRL_HISTORY);
    if(e==cudaSuccess) e = cudaFuncSetAttribute(pcm16x0_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227*1024);
    if(e==cudaSuccess) e = cudaMalloc(&h->p1_stats_dev, 4*sizeof(unsigned long long));
    if(e==cudaSuccess) e = cudaMallocHost(&h->p1_stats_host, 4*sizeof(unsigned long long));
    if(e!=cudaSuccess) { sdv_destroy(h); return SDV_ERR_CUDA; }
    *out = h;
    return SDV_OK;
}

void sdv_destroy(sdv_handle *h)
{
    if(!h) return;
    cudaSetDevice(h->device);
    cudaFree(h->ctx); cudaFree(h->clean); cudaFree(h->bits); cudaFree(h->seg_ctx); cudaFree(h->pad_dev);
    cudaFree(h->x0_scan); cudaFree(h->x0_scan_ei); cudaFree(h->x0_geo); cudaFree(h->x0_mask);
    cudaFree(h->snaps); cudaFree(h->start_ctx); cudaFree(h->fmed); cudaFree(h->warm_scratch); cudaFree(h->relay_ok); cudaFreeHost(h->relay_ok_host);
    cudaFree(h->win_state); cudaFreeHost(h->win_state_host); cudaFree(h->trim_dev); cudaFree(h->fa_dev); cudaFree(h->task_dev); cudaFree(h->sstat_dev);
    for(int i=0;i<2;i++) { cudaFree(h->carry_dev[i]); cudaFree(h->carry_meta_dev[i]); cudaFree(h->cwd_carry[i]); }
    cudaFree(h->cwd_spec_dev); cudaFree(h->cwd_status); cudaFree(h->cwd_scan_dev); cudaFree(h->cwd_plan_dev); cudaFree(h->blk_scratch); cudaFree(h->fres_dev);
    cudaFree(h->luma_dev); cudaFree(h->recs_dev); cudaFree(h->smp_dev); cudaFree(h->sfl_dev);
    cudaFreeHost(h->hdr_host); cudaFreeHost(h->fu_host); cudaFree(h->spec_fu);
    cudaFree(h->p1_scan); cudaFree(h->p1_presets); cudaFree(h->p1_clean); cudaFree(h->p1_bw); cudaFree(h->p1_ctx); cudaFree(h->x0_ctx); cudaFree(h->x0_votes);
    cudaFree(h->p1_stats_dev); cudaFreeHost(h->p1_stats_host); cudaFree(h->p1_sub);
    for(int i=0;i<2;i++) if(h->ev_sync[i]) cudaEventDestroy(h->ev_sync[i]);
    if(h->ev_lazy) cudaEventDestroy(h->ev_lazy);
    if(h->stream) cudaStreamDestroy(h->stream);
    if(h->copy_stream) cudaStreamDestroy(h->copy_stream);
    for(int i=0;i<4;i++) if(h->ev[i]) cudaEventDestroy(h->ev[i]);
    delete h;
}

// Fold the device time of the last bulk (which = 0) / deinterleave (which = 1) launch into the accumulators.
static void timing_flush(sdv_handle *h, int which)
{
    if(!h->ev_set[which]) return;
    float ms = 0;
    if((cudaEventSynchronize(h->ev[2*which+1])==cudaSuccess)&&(cudaEventElapsedTime(&ms, h->ev[2*which], h->ev[2*which+1])==cudaSuccess))
    {
        h->acc_ms[which] += ms; h->acc_units[which] += h->ev_units[which]; h->acc_n[which]++;
    }
    h->ev_set[which] = 0;
}

static int ensure(sdv_handle *h, void **p, size_t *cap, size_t need)
{
    if(*cap>=need) return SDV_OK;
    if(*p) { cudaFree(*p); *p = NULL; *cap = 0; }
    cudaError_t e = cudaMalloc(p, need);
    if(e!=cudaSuccess) return fail(h, SDV_ERR_NOMEM, "cudaMalloc", e);
    *cap = need;
    return SDV_OK;
}

static int read_hdr(sdv_handle *h, cudaStream_t st)
{
    CK(cudaMemcpyAsync(h->hdr_host, h->ctx, sizeof(ChainHdr), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SDV_OK;
}

// PCM-1: prescan of every frame -> per-frame presets -> bulk pass -> chain (pcm1_kernels.cuh).  Four launches, one sync.
static int p1_decode_frames(sdv_handle *h, const sdv_bin_config *cfg, const uint8_t *luma_dev, int n_frames, int H, int W,
                            int stride, sdv_line_rec *recs_dev, sdv_line_aux *aux_dev, cudaStream_t st)
{
    const bool x0 = (cfg->pcm_type==SDV_TYPE_PCM16X0);      // PCM-16x0: three sub-line records per video line
    if(W<(x0 ? (int)X0L_BITS : (int)P1_BITS)) return fail(h, SDV_ERR_ARG, "line shorter than the PCM bit cells", cudaSuccess);
    // reserved[3] bit 0: this call continues the file of the previous PCM call on the handle: the chain state in p1_ctx / x0_ctx
    // (Binarizer presets, coordinate histories, prescan_ref, the running pair G) goes on, and frame 0 is not the file's first
    const int key_mode = cfg->mode|((cfg->check_line_dup ? 1 : 0)<<8);
    const bool cont = (cfg->reserved[3]&1)!=0;
    if(cont&&!(h->pcm_open&&(h->pcm_type==cfg->pcm_type)&&(h->pcm_H==H)&&(h->pcm_W==W)&&(h->pcm_mode==key_mode)))
        return fail(h, SDV_ERR_ARG, "sdv_bin_decode_frames: nothing to continue (no earlier call with this PCM type, geometry and mode on the handle)", cudaSuccess);
    if(cont&&(((int)cfg->reserved[0]|((int)cfg->reserved[1]<<8))>1))
        return fail(h, SDV_ERR_ARG, "sdv_bin_decode_frames: a continuing PCM-1 / PCM-16x0 call decodes one file (chain_segments must be 0 or 1)", cudaSuccess);
    h->pcm_open = 0;
    int rc;
    if((rc = ensure(h, (void **)&h->p1_scan, &h->p1_scan_cap, (size_t)n_frames*P1_COORD_CHECK_LINES*sizeof(P1Preset)))) return rc;
    if((rc = ensure(h, (void **)&h->p1_presets, &h->p1_presets_cap, (size_t)n_frames*sizeof(P1Preset)))) return rc;
    if((rc = ensure(h, (void **)&h->p1_clean, &h->p1_clean_cap, (size_t)n_frames+16))) return rc;
    if((rc = ensure(h, (void **)&h->p1_bw, &h->p1_bw_cap, (size_t)n_frames*sizeof(u32)))) return rc;
    const bool prescan = (cfg->mode!=SDV_MODE_DRAFT);
    if(prescan)
    {
        if(x0) pcm16x0_prescan_kernel<<<n_frames*P1_COORD_CHECK_LINES, P1S_THREADS, 0, st>>>(luma_dev, H, W, (size_t)stride, n_frames, cfg->mode, !cont, h->p1_scan);
        else pcm1_prescan_kernel<<<n_frames*P1_COORD_CHECK_LINES, P1S_THREADS, 0, st>>>(luma_dev, H, W, (size_t)stride, n_frames, cfg->mode, !cont, h->p1_scan);
        h->stats.kernel_launches++;
    }
    pcm1_preset_kernel<<<(n_frames+255)/256, 256, 0, st>>>(h->p1_scan, n_frames, H, cfg->mode, !cont, h->p1_presets);
    h->stats.kernel_launches++;
    // bulk pass (only meaningful with per-frame presets, i.e. when the prescan runs)
    const BulkPlan bulk = bulk_plan(W, stride, luma_dev, P1_BULK_HEADER);
    // the bulk pass knows the first-line rule of the duplicate-line check at its default only (en_first_line_dup): with the switch
    // off every frame goes through the chain kernel
    const bool use_bulk = prescan&&(bulk.warps>=1)&&(H>=2*BULK_ROWS)&&p1_prescan_runs(H, false, cfg->mode)
                          &&(h->fine.en_first_line_dup||!cfg->check_line_dup);
    if(use_bulk)
    {
        P1BulkParams bp;
        bp.luma = luma_dev; bp.H = H; bp.W = W; bp.stride = (size_t)stride; bp.n_frames = n_frames;
        bp.presets = h->p1_presets; bp.run_g = (x0&&cont) ? &h->x0_ctx->run_g : h->p1_presets; bp.line_dup = cfg->check_line_dup ? 1 : 0; bp.mode = cfg->mode;
        bp.recs = recs_dev; bp.aux = aux_dev; bp.clean = h->p1_clean; bp.frame_bw = h->p1_bw;
        bp.use_tma = bulk.use_tma; bp.warps = bulk.warps; bp.slot_bytes = bulk.slot_bytes;
        int grid = (n_frames+bulk.warps-1)/bulk.warps;
        if(grid>h->num_sms) grid = h->num_sms;
        timing_flush(h, 0);
        cudaEventRecord(h->ev[0], st);
        if(x0) pcm16x0_bulk_kernel<<<grid, bulk.warps*32, bulk.smem, st>>>(bp);
        else pcm1_bulk_kernel<<<grid, bulk.warps*32, bulk.smem, st>>>(bp);
        cudaEventRecord(h->ev[1], st);
        h->ev_set[0] = 1; h->ev_units[0] = (uint64_t)n_frames*(uint64_t)H;
        h->stats.kernel_launches++;
    }
    if(x0)
    {
        X0ChainParams xp;
        xp.luma = luma_dev; xp.H = H; xp.W = W; xp.stride = (size_t)stride; xp.n_frames = n_frames;
        xp.mode = cfg->mode; xp.line_dup = cfg->check_line_dup ? 1 : 0; xp.use_bulk = use_bulk ? 1 : 0; xp.cont = cont ? 1 : 0;
        xp.scan = h->p1_scan; xp.presets = h->p1_presets; xp.clean = h->p1_clean; xp.frame_bw = h->p1_bw;
        xp.recs = recs_dev; xp.aux = aux_dev; xp.ctx = h->x0_ctx; xp.stats = h->p1_stats_dev;
        pcm16x0_chain_kernel<<<1, P1L_THREADS, sizeof(X0ChainCtx), st>>>(xp);
    }
    else
    {
    P1ChainParams cp;
    cp.luma = luma_dev; cp.H = H; cp.W = W; cp.stride = (size_t)stride; cp.n_frames = n_frames;
    cp.mode = cfg->mode; cp.line_dup = cfg->check_line_dup ? 1 : 0; cp.use_bulk = use_bulk ? 1 : 0; cp.cont = cont ? 1 : 0;
    cp.presets = h->p1_presets; cp.clean = h->p1_clean; cp.frame_bw = h->p1_bw;
    cp.recs = recs_dev; cp.aux = aux_dev; cp.ctx = h->p1_ctx; cp.stats = h->p1_stats_dev;
    pcm1_chain_kernel<<<1, P1L_THREADS, sizeof(P1ChainCtx), st>>>(cp);
    }
    h->stats.kernel_launches++;
    CK(cudaMemcpyAsync(h->p1_stats_host, h->p1_stats_dev, 4*sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    h->stats.lines_chain = h->p1_stats_host[0];
    h->stats.frames_skipped = h->p1_stats_host[2];
    h->stats.reserved = (uint32_t)h->p1_stats_host[3];      // (sub-)lines the chain kernel took from the bulk pass as hints
    h->stats.lines_fast = h->p1_stats_host[2]*(uint64_t)H*(x0 ? 3 : 1);
    if(x0) h->stats.lines_total = (uint64_t)n_frames*H*3;
    h->acc_launches += h->stats.kernel_launches;
    h->pcm_open = 1; h->pcm_type = cfg->pcm_type; h->pcm_H = H; h->pcm_W = W; h->pcm_mode = key_mode;
    return SDV_OK;
}

static int decode_frames_impl(sdv_handle *h, const sdv_bin_config *cfg, const uint8_t *luma_dev, int n_frames, int H, int W,
                              int stride, sdv_line_rec *recs_dev, sdv_line_aux *aux_dev, void *cuda_stream);
struct DeintScratch { u32 *bits; u8 *sum; WindowList wl; };
static int deint_scratch(sdv_handle *h, long long n_blocks, int dur, DeintScratch *o)
{
    const size_t words = (size_t)((n_blocks+31)>>5), groups = (size_t)((n_blocks+1023)>>10);
    const size_t cap = (dur>0) ? (size_t)(n_blocks/dur+2) : 1;
    const size_t o_sum = words*sizeof(u32), o_start = (o_sum+groups+15)&~(size_t)15, o_len = o_start+cap*sizeof(long long);
    int rc = ensure(h, (void **)&h->bits, &h->bits_cap, o_len+cap*sizeof(int)+64);
    if(rc) return rc;
    u8 *base = (u8 *)h->bits;
    o->bits = h->bits; o->sum = base+o_sum;
    o->wl.start = (long long *)(base+o_start); o->wl.len = (int *)(base+o_len); o->wl.cap = (int)((cap>0x7FFFFFFF) ? 0x7FFFFFFF : cap); o->wl.state = h->win_state;
    return SDV_OK;
}

// ---- fine settings.  The device code reads them from one __constant__ object per device; a decode call whose handle holds
// other values than the object waits for the device to drain and rewrites it (handles with different settings can share a
// device, they just do not overlap).
static std::mutex g_fine_mtx;
static FineSet g_fine_cur[64];
static bool g_fine_init = false;
static bool fine_equal(const FineSet &a, const FineSet &b) { return memcmp(&a, &b, sizeof(FineSet))==0; }
static int apply_fine(sdv_handle *h)
{
    std::lock_guard<std::mutex> lk(g_fine_mtx);
    if(!g_fine_init) { const FineSet d = SDV_FINE_DEFAULTS; for(int i=0;i<64;i++) g_fine_cur[i] = d; g_fine_init = true; }
    const int dev = h->device&63;
    if(fine_equal(g_fine_cur[dev], h->fine)) return SDV_OK;
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyToSymbol(c_fine, &h->fine, sizeof(FineSet)));
    CK(cudaDeviceSynchronize());
    g_fine_cur[dev] = h->fine;
    return SDV_OK;
}
int sdv_bin_default_fine_settings(sdv_bin_preset *out)
{
    if(!out) return SDV_ERR_ARG;
    memset(out, 0, sizeof(*out));
    const FineSet d = SDV_FINE_DEFAULTS;
    out->max_black_lvl = d.max_black_lvl; out->min_white_lvl = d.min_white_lvl; out->min_contrast = d.min_contrast;
    out->min_ref_lvl = d.min_ref_lvl; out->max_ref_lvl = d.max_ref_lvl; out->min_valid_crcs = d.min_valid_crcs;
    out->mark_max_dist = d.mark_max_dist; out->left_bit_pick = d.left_bit_pick; out->right_bit_pick = d.right_bit_pick;
    out->en_force_coords = 0; out->en_coord_search = 1; out->en_first_line_dup = 1; out->en_good_no_marker = 1;
    return SDV_OK;
}
int sdv_bin_get_fine_settings(sdv_handle *h, sdv_bin_preset *out)
{
    if(!h||!out) return SDV_ERR_ARG;
    sdv_bin_default_fine_settings(out);
    const FineSet &d = h->fine;
    out->max_black_lvl = d.max_black_lvl; out->min_white_lvl = d.min_white_lvl; out->min_contrast = d.min_contrast;
    out->min_ref_lvl = d.min_ref_lvl; out->max_ref_lvl = d.max_ref_lvl; out->min_valid_crcs = d.min_valid_crcs;
    out->mark_max_dist = d.mark_max_dist; out->left_bit_pick = d.left_bit_pick; out->right_bit_pick = d.right_bit_pick;
    out->en_coord_search = d.en_coord_search; out->en_first_line_dup = d.en_first_line_dup;
    return SDV_OK;
}
int sdv_bin_set_fine_settings(sdv_handle *h, const sdv_bin_preset *in)
{
    if(!h||!in) return SDV_ERR_ARG;
    if(in->en_force_coords||!in->en_good_no_marker)
        return fail(h, SDV_ERR_UNSUPPORTED, "sdv_bin_set_fine_settings: en_force_coords / en_good_no_marker are taken at their defaults only (0, 1)", cudaSuccess);
    if((in->left_bit_pick>4)||(in->right_bit_pick>2)||(in->mark_max_dist>50)||(in->min_ref_lvl>in->max_ref_lvl))
        return fail(h, SDV_ERR_ARG, "sdv_bin_set_fine_settings: left_bit_pick <= 4, right_bit_pick <= 2, mark_max_dist <= 50, min_ref_lvl <= max_ref_lvl", cudaSuccess);
    FineSet f; memset(&f, 0, sizeof(f));
    f.max_black_lvl = in->max_black_lvl; f.min_white_lvl = in->min_white_lvl; f.min_contrast = in->min_contrast;
    f.min_ref_lvl = in->min_ref_lvl; f.max_ref_lvl = in->max_ref_lvl; f.min_valid_crcs = in->min_valid_crcs;
    f.mark_max_dist = in->mark_max_dist; f.left_bit_pick = in->left_bit_pick; f.right_bit_pick = in->right_bit_pick;
    f.en_coord_search = in->en_coord_search ? 1 : 0; f.en_first_line_dup = in->en_first_line_dup ? 1 : 0;
    if(!fine_equal(f, h->fine)) { h->fine = f; h->warm_valid = 0; h->chain_open = 0; h->pcm_open = 0; }     // presets found with other settings are no guess for these
    return SDV_OK;
}

int sdv_bin_on_first_frame(sdv_handle *h, sdv_first_frame_fn fn, void *user)
{
    if(!h) return SDV_ERR_ARG;
    h->first_frame_fn = fn; h->first_frame_user = user;
    return SDV_OK;
}

int sdv_bin_decode_frames(sdv_handle *h, const sdv_bin_config *cfg, const uint8_t *luma_dev, int n_frames, int H, int W,
                          int stride, sdv_line_rec *recs_dev, sdv_line_aux *aux_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    h->first_frame_called = 0;
    const int rc = decode_frames_impl(h, cfg, luma_dev, n_frames, H, W, stride, recs_dev, aux_dev, cuda_stream);
    if((rc==SDV_OK)&&h->first_frame_fn&&!h->first_frame_called) { h->first_frame_called = 1; h->first_frame_fn(h->first_frame_user); }   // no early point on this path
    return rc;
}

static int decode_frames_impl(sdv_handle *h, const sdv_bin_config *cfg, const uint8_t *luma_dev, int n_frames, int H, int W,
                              int stride, sdv_line_rec *recs_dev, sdv_line_aux *aux_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!cfg||(n_frames<0)||(H<2)||(H&1)||(H>SDV_MAX_H)||(W<BITS_IN_LINE)||(W>SDV_MAX_W)||(stride<W))     // the chain keeps one coordinate pair per line of a frame (SDV_MAX_H of them)
        return fail(h, SDV_ERR_ARG, "sdv_bin_decode_frames: frame geometry (2 <= H <= 1250 even, 137 <= W <= 2048, stride >= W)", cudaSuccess);
    if((n_frames>0)&&(!luma_dev||!recs_dev||((uintptr_t)recs_dev%16)||((uintptr_t)aux_dev%16)))
        return fail(h, SDV_ERR_ARG, "sdv_bin_decode_frames: null or misaligned buffer (records need 16-byte alignment)", cudaSuccess);
    if((cfg->pcm_type!=SDV_TYPE_STC007)&&(cfg->pcm_type!=SDV_TYPE_PCM1)&&(cfg->pcm_type!=SDV_TYPE_PCM16X0)&&(cfg->pcm_type!=SDV_TYPE_M2))
        return fail(h, SDV_ERR_UNSUPPORTED, "pcm_type", cudaSuccess);
    const int dup_flags = (cfg->check_line_dup ? 1 : 0)|((cfg->pcm_type==SDV_TYPE_M2) ? 2 : 0);     // chain_reset / BulkParams packing
    if(cfg->mode>SDV_MODE_INSANE) return fail(h, SDV_ERR_ARG, "mode", cudaSuccess);
    CK(cudaSetDevice(h->device));
    if(h->lazy_pending) return fail(h, SDV_ERR_ARG, "sdv_bin_decode_frames: the previous call was lazy (reserved[2] bit 1): call sdv_bin_decode_verify first", cudaSuccess);
    { const int frc = apply_fine(h); if(frc) return frc; }
    cudaStream_t st = (cudaStream_t)cuda_stream;
    memset(&h->stats, 0, sizeof(h->stats));
    h->stats.lines_total = (uint64_t)n_frames*H;
    if(n_frames==0) return SDV_OK;
    if((cfg->pcm_type==SDV_TYPE_PCM1)||(cfg->pcm_type==SDV_TYPE_PCM16X0)) return p1_decode_frames(h, cfg, luma_dev, n_frames, H, W, stride, recs_dev, aux_dev, st);
    { int rc = ensure(h, (void **)&h->clean, &h->clean_cap, 2*(size_t)n_frames+16); if(rc) return rc; }


    const BulkPlan bulk = bulk_plan(W, stride, luma_dev, BULK_SMEM_HEADER);
    if(bulk.warps<1) return fail(h, SDV_ERR_ARG, "line too wide for the bulk kernel", cudaSuccess);

    // Segment mode: the tape is decoded as [chain_segments] independent files, one chain per thread block, all in
    // one launch.  For tapes whose lines keep failing the preset decode (every frame would go through the single
    // sequential chain otherwise).  Each segment equals the reference run on that piece of tape.
    int segments = (int)cfg->reserved[0]|((int)cfg->reserved[1]<<8);
    if(segments>n_frames) segments = n_frames;
    if(segments>1)
    {
        h->fuse_arm.armed = 0; h->fuse_done.valid = 0;
        if(h->seg_cap<(size_t)segments)
        {
            cudaFree(h->seg_ctx); h->seg_ctx = NULL; h->seg_cap = 0;
            CK(cudaMalloc(&h->seg_ctx, (size_t)segments*sizeof(ChainCtx)));
            h->seg_cap = (size_t)segments;
        }
        ChainParams cp; memset(&cp, 0, sizeof(cp));
        cp.luma = luma_dev; cp.H = H; cp.W = W; cp.stride = (size_t)stride;
        cp.f_begin = 0; cp.n_frames = n_frames; cp.max_frames = n_frames;
        cp.recs = recs_dev; cp.aux = aux_dev; cp.ctx = h->seg_ctx;
        cp.clean = NULL; cp.have_spec = 0; cp.spec_ref = 0; cp.spec_coords = coord_none();
        cp.reset = 1; cp.mode = cfg->mode; cp.line_dup = dup_flags; cp.segments = segments;
        stc007_chain_kernel<256><<<segments, 256, 0, st>>>(cp);
        h->stats.kernel_launches++;
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
        h->stats.lines_chain = h->stats.lines_total;
        h->acc_launches += h->stats.kernel_launches;
        return SDV_OK;
    }

    // reserved[3] bit 0: this call continues the file of the previous sdv_bin_decode_frames call on the handle: the chain
    // (Binarizer presets, coordinate histories, videotodigital.cpp:707-710,1366-1522) goes on from where that call left it
    const bool cont = (cfg->reserved[3]&1)&&h->chain_open&&(h->chain_H==H)&&(h->chain_W==W)&&(h->chain_mode==(cfg->mode|(dup_flags<<8)));
    if((cfg->reserved[3]&1)&&!cont) return fail(h, SDV_ERR_ARG, "sdv_bin_decode_frames: nothing to continue (no earlier call with this geometry and mode on the handle)", cudaSuccess);
    h->chain_open = 0;
    int f = 0;
    bool have_spec = false; u8 spec_ref = 0, spec_black = 0, spec_white = 0; Coord spec_c = coord_none();
    uint64_t frames_bulk = 0;
    // Fused deinterleave (sdv_stc007_fuse_next_decode): the bulk pass also finishes the data blocks that lie inside a frame.  It
    // counts only if ONE bulk launch ends up supplying every frame behind its first one; else the deinterleave call does all blocks.
    const bool fuse_req = h->fuse_arm.armed&&(cfg->pcm_type==SDV_TYPE_STC007)&&(H/2<=BULK_FUSE_HF)&&(H/2<=h->fuse_arm.geo.lines_per_field)&&!cont;
    h->fuse_arm.armed = 0; h->fuse_done.valid = 0;
    int fuse_launches = 0, fuse_from = 0; bool fuse_ok = fuse_req;
    DeintScratch fsc; memset(&fsc, 0, sizeof(fsc));
    long long fuse_blocks = 0;
    if(fuse_req)
    {
        fuse_blocks = (long long)h->fuse_arm.geo.lead_in+(long long)n_frames*2*h->fuse_arm.geo.lines_per_field;
        const int rc = deint_scratch(h, fuse_blocks, h->fuse_arm.cfg.broken_mask_dur, &fsc);
        if(rc) return rc;
    }

    // Persistent grid, one block per SM, but not on every SM.  Measured on B200 at 720 px lines (profiles/r1_bulk_grid_sweep.md):
    // the pass scales linearly with the block count up to ~130 blocks (each SM is issue-bound at ~52 GB/s), reaches ~7.0 TB/s
    // there, and gets SLOWER beyond it (-5% at 134, 6.2 TB/s at 148) as HBM is oversubscribed; 0.88 x SMs sits just left of that edge.  The SMs left over also give the
    // 1024-thread chain block that runs beside the speculative pass a home: it needs a whole SM's registers and would
    // otherwise wait for the first bulk block to retire.  SDV_BULK_BLOCKS overrides the count (tuning knob).
    static const int bulk_blocks_env = getenv("SDV_BULK_BLOCKS") ? atoi(getenv("SDV_BULK_BLOCKS")) : 0;
    const int bulk_blocks = (bulk_blocks_env>0) ? ((bulk_blocks_env<h->num_sms) ? bulk_blocks_env : h->num_sms)
                                                : ((h->num_sms>8) ? (h->num_sms*88)/100 : h->num_sms);
    auto launch_bulk = [&](cudaStream_t bst, int f_from, const BinState &b, int *first_unclean_dev)
    {
        BulkParams bp;
        bp.luma = luma_dev; bp.H = H; bp.W = W; bp.stride = (size_t)stride;
        bp.f0 = f_from; bp.n_frames = n_frames-f_from;
        bp.ref = b.def_ref; bp.black = b.def_black; bp.white = b.def_white; bp.line_dup = (u8)dup_flags; bp.coords = b.def_coord;
        bp.recs = recs_dev; bp.aux = aux_dev; bp.clean = h->clean; bp.first_unclean = first_unclean_dev;
        bp.use_tma = bulk.use_tma; bp.slot_bytes = bulk.slot_bytes;
        { const Ppb ppb = make_ppb(b.def_coord); for(int i=0;i<BITS_PCM_DATA;i++) bp.pos[i] = (u32)pixel_of_bit(ppb, i, 0, W-1); }
        const long long units = (long long)(n_frames-f_from);      // frames
        const bool fuse = fuse_req&&(fuse_launches==0);
        BulkPlan pl = bulk;
        if(fuse)
        {   // the same slots, with room for the line words of one frame per warp
            const BulkPlan fp = bulk_plan_warps(bulk, BULK_SMEM_HEADER, BULK_FUSE_BYTES);
            if(fp.warps<1) fuse_ok = false;
            else pl = fp;
        }
        const bool fuse_now = fuse&&fuse_ok;
        bp.warps = pl.warps;
        bp.samples = NULL; bp.sflags = NULL; bp.broken_bits = NULL; bp.broken_sum = NULL; bp.block0 = 0; bp.lpf = 0;
        if(fuse_now)
        {
            bp.samples = h->fuse_arm.samples; bp.sflags = h->fuse_arm.sflags;
            bp.broken_bits = fsc.bits; bp.broken_sum = fsc.sum;
            bp.block0 = h->fuse_arm.geo.lead_in; bp.lpf = h->fuse_arm.geo.lines_per_field;
            cudaMemsetAsync(fsc.bits, 0, (size_t)((fuse_blocks+31)>>5)*sizeof(u32)+(size_t)((fuse_blocks+1023)>>10), bst);
            fuse_from = f_from;
        }
        else if(fuse_req) fuse_ok = false;                          // a second bulk launch: its frames are not fused
        fuse_launches++;
        int grid = (int)((units+pl.warps-1)/pl.warps);
        // the fused pass carries ~10 % more instructions per line: every SM but the one the first-frame chain block needs
        const int max_blocks = (fuse_now&&(bulk_blocks_env<=0)&&(h->num_sms>8)) ? (h->num_sms-1) : bulk_blocks;
        if(grid>max_blocks) grid = max_blocks;
        timing_flush(h, 0);
        cudaEventRecord(h->ev[0], bst);
        if(fuse_now) stc007_bulk_kernel<true><<<grid, pl.warps*32, pl.smem, bst>>>(bp);
        else stc007_bulk_kernel<false><<<grid, pl.warps*32, pl.smem, bst>>>(bp);
        cudaEventRecord(h->ev[1], bst);
        h->ev_set[0] = 1; h->ev_units[0] = (uint64_t)(n_frames-f_from)*(uint64_t)H;
        h->stats.kernel_launches++;
    };

    // Warm start: the steady-state presets the previous decode of this handle ended with are the best guess for this one
    // (consecutive pieces of a capture share levels and geometry).  The bulk kernel is launched with them on a second
    // stream, concurrently with the chain kernel that derives the true presets from the first frame; the guess is kept
    // only if the chain kernel arrives at exactly the same presets after exactly one frame, otherwise everything is
    // redone without it.  Scheduling only: results never depend on the guess.  Not on a call that continues the file: its chain
    // kernel advances the file's chain state in place, so a wrong guess could not start the call over from that state.
    bool warm_pending = false;
    if(h->warm_valid&&(h->warm_H==H)&&(h->warm_W==W)&&(h->warm_mode==(cfg->mode|(dup_flags<<8)))&&(n_frames>1)&&!(cfg->reserved[2]&1)&&!cont)
    {
        CK(cudaEventRecord(h->ev_sync[0], st));
        CK(cudaStreamWaitEvent(h->copy_stream, h->ev_sync[0], 0));
        set_int_kernel<<<1, 1, 0, h->copy_stream>>>(h->spec_fu, n_frames);
        launch_bulk(h->copy_stream, 1, h->warm_bin, h->spec_fu);
        CK(cudaEventRecord(h->ev_sync[1], h->copy_stream));
        warm_pending = true;
    }
    // Relay mode (frames [f0, n_frames) of a tape whose chain does not settle): exactly the single sequential chain of
    // the reference, computed by many chains at once.  The frames are cut into pieces, one thread block each.  A piece
    // needs the chain state at its head, which only the pieces before it can give -- so it is guessed: the block decodes
    // the RELAY_WARM frames before its piece from an empty state (that rebuilds the presets and the last-9-lines history)
    // with the 16-frame coordinate history seeded from the per-frame medians of a first pass.  Afterwards piece b is kept
    // only if its guessed start state EQUALS the end state of piece b-1 (chain_state_equal): by induction from piece 0,
    // which starts from the true state, every kept piece is what the sequential chain produces.  A piece that fails the
    // test is decoded again from the true state by the sequential kernel (and the test repeated for the next one).
    enum { RELAY_AFTER = 2, RELAY_MIN_FRAMES = 32, RELAY_WARM = 2, RELAY_LEN = 2, CHAIN_LAUNCH_FRAMES = 64 };
    int chain_run = 0;              // frames in a row decoded by the chain kernel, none taken from the bulk pass in between
    bool relayed = false;
    int relay_end = 0, relay_pieces = 0, relay_redone = 0;
    auto relay_decode = [&](int f0) -> int
    {
        // one round covers what the device holds at once (four 256-thread chains per SM, RELAY_LEN frames each); a longer tape
        // goes back to the ordinary loop afterwards, which hands clean stretches to the bulk pass again
        static const int len_env = getenv("SDV_RELAY_LEN") ? atoi(getenv("SDV_RELAY_LEN")) : 0;      // tuning knob
        const int len = (len_env>0) ? len_env : RELAY_LEN;
        const int span = (n_frames-f0<4*h->num_sms*len) ? (n_frames-f0) : (4*h->num_sms*len);
        const int left = span;
        const int pieces = (left+len-1)/len;
        const int n_frames_all = n_frames;
        const int n_frames = f0+span;          // (shadows the tape length inside this round)
        (void)n_frames_all;
        relay_end = n_frames;
        int rc;
        if(h->seg_cap<(size_t)pieces)
        {
            cudaFree(h->seg_ctx); h->seg_ctx = NULL; h->seg_cap = 0;
            CK(cudaMalloc(&h->seg_ctx, (size_t)pieces*sizeof(ChainCtx)));
            h->seg_cap = (size_t)pieces;
        }
        if((rc = ensure(h, (void **)&h->start_ctx, &h->start_cap, (size_t)pieces*sizeof(ChainCtx)))) return rc;
        if((rc = ensure(h, (void **)&h->fmed, &h->fmed_cap, 2*(size_t)n_frames_all*sizeof(Coord)))) return rc;
        if((rc = ensure(h, (void **)&h->snaps, &h->snaps_cap, (size_t)n_frames_all*sizeof(ChainSnap)))) return rc;
        if((rc = ensure(h, (void **)&h->warm_scratch, &h->warm_cap, (size_t)pieces*CHAIN_BATCH*sizeof(sdv_line_rec)))) return rc;
        if((rc = ensure(h, (void **)&h->relay_ok, &h->relay_ok_cap, (size_t)pieces*(1+sizeof(int))+32))) return rc;
        if(h->relay_ok_host_cap<(size_t)pieces)
        {
            cudaFreeHost(h->relay_ok_host); h->relay_ok_host = NULL; h->relay_ok_host_cap = 0;
            CK(cudaMallocHost(&h->relay_ok_host, (size_t)pieces));
            h->relay_ok_host_cap = (size_t)pieces;
        }
        static const bool trace = getenv("SDV_RELAY_TRACE")!=NULL;
        auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        double t_mark = 0;
        if(trace) { cudaStreamSynchronize(st); t_mark = now(); fprintf(stderr, "[relay] from frame %d, %d pieces of %d frames\n", f0, pieces, len); }
        Coord *fm_a = h->fmed, *fm_b = h->fmed+n_frames_all;
        seed_fmed_kernel<<<(unsigned)((n_frames+255)/256), 256, 0, st>>>(h->ctx, fm_a, f0, n_frames);
        ChainParams rp; memset(&rp, 0, sizeof(rp));
        rp.luma = luma_dev; rp.H = H; rp.W = W; rp.stride = (size_t)stride;
        rp.f_begin = f0; rp.n_frames = n_frames; rp.max_frames = n_frames;
        rp.recs = recs_dev; rp.aux = aux_dev; rp.ctx = h->seg_ctx; rp.spec_coords = coord_none();
        rp.mode = cfg->mode; rp.line_dup = dup_flags; rp.segments = 1; rp.cont = cont ? 1 : 0;
        rp.relay_len = len; rp.relay_warm = RELAY_WARM; rp.start_ctx = h->start_ctx; rp.warm_scratch = h->warm_scratch; rp.snaps = h->snaps;
        // Pass 0: every piece decoded from its guessed state, guessing that the 16-frame coordinate history stays what it is.
        // Then, while pieces fail the test: the failing pieces are guessed afresh with the history taken from the medians the
        // decode has found so far (a frame whose median moved spoils the guess of the 16 frames behind it) -- or, once that
        // stops paying, decoded from the end state of the piece before them, which is right for the leftmost piece of every
        // run of failing pieces in each round (and for the others as soon as the piece before them comes out unchanged).
        CK(cudaMemcpyAsync(h->seg_ctx, h->ctx, sizeof(ChainCtx), cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(fm_b, fm_a, (size_t)n_frames*sizeof(Coord), cudaMemcpyDeviceToDevice, st));
        rp.fmed_in = fm_a; rp.fmed_out = fm_b;
        stc007_chain_kernel<256><<<pieces, 256, 0, st>>>(rp);
        h->stats.kernel_launches++;
        { Coord *t = fm_a; fm_a = fm_b; fm_b = t; }
        int redone = 0, reseeds = 0, last_bad = pieces+1;
        std::vector<int> list;
        int *const list_dev = (int *)(h->relay_ok+(((size_t)pieces+15)&~(size_t)15));      // behind the flags
        static const int reseed_env = getenv("SDV_RELAY_RESEED") ? atoi(getenv("SDV_RELAY_RESEED")) : 0;     // tuning knob (measured on BASELINE config 4: re-guessing does not pay, profiles/r2_config4_relay.md)
        for(int round=0;round<=2*pieces+8;round++)
        {
            chain_verify_kernel<<<(unsigned)((pieces+255)/256), 256, 0, st>>>(h->start_ctx, h->seg_ctx, pieces, h->relay_ok);
            CK(cudaMemcpyAsync(h->relay_ok_host, h->relay_ok, (size_t)pieces, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            h->stats.kernel_launches++;
            list.clear();
            int longest = 0;
            for(int b=1, run=0;b<pieces;b++) { if(!h->relay_ok_host[b]) { list.push_back(b); run++; if(run>longest) longest = run; } else run = 0; }
            if(trace) { const double t = now(); fprintf(stderr, "[relay] round %d: %.1f ms, %d pieces fail the test, longest run %d\n", round, t-t_mark, (int)list.size(), longest); t_mark = t; }
            if(list.empty()) break;
            CK(cudaMemcpyAsync(list_dev, list.data(), list.size()*sizeof(int), cudaMemcpyHostToDevice, st));
            rp.relay_list = list_dev;
            const bool reseed = (reseeds<reseed_env)&&(longest>2)&&((int)list.size()<last_bad);
            last_bad = (int)list.size();
            if(reseed)
            {
                CK(cudaMemcpyAsync(fm_b, fm_a, (size_t)n_frames*sizeof(Coord), cudaMemcpyDeviceToDevice, st));
                rp.fmed_in = fm_a; rp.fmed_out = fm_b;
                reseeds++;
            }
            else { rp.fmed_in = NULL; rp.fmed_out = fm_a; }
            if((int)list.size()<=h->num_sms) stc007_chain_kernel<1024><<<(unsigned)list.size(), 1024, 0, st>>>(rp);     // room for a whole SM each
            else stc007_chain_kernel<256><<<(unsigned)list.size(), 256, 0, st>>>(rp);
            if(reseed) { Coord *t = fm_a; fm_a = fm_b; fm_b = t; }
            h->stats.kernel_launches++;
            redone += (int)list.size();
        }
        CK(cudaMemcpyAsync(h->ctx, h->seg_ctx+(pieces-1), sizeof(ChainCtx), cudaMemcpyDeviceToDevice, st));
        { int rc2 = read_hdr(h, st); if(rc2) return rc2; }
        h->stats.frames_skipped = 0;
        relay_pieces += pieces; relay_redone += redone;
        h->stats.reserved = (uint32_t)(((uint32_t)((relay_pieces>0xFFFF) ? 0xFFFF : relay_pieces)<<16)|(uint32_t)((relay_redone>0xFFFF) ? 0xFFFF : relay_redone));     // relay: pieces | pieces decoded again
        return SDV_OK;
    };
    while(f<n_frames)
    {
        if((chain_run>=RELAY_AFTER)&&(n_frames-f>=RELAY_MIN_FRAMES)&&!(cfg->reserved[2]&4)&&!warm_pending)
        {   // RELAY_AFTER frames in a row that the bulk pass could not take: a damaged tape, the rest goes in relay mode
            fuse_ok = false;
            const int rc = relay_decode(f);
            if(rc) return rc;
            f = relay_end;
            relayed = true;
            chain_run = 0;
            have_spec = false;          // the bulk records behind f (if any) were overwritten
            continue;
        }
        ChainParams cp; memset(&cp, 0, sizeof(cp));
        cp.luma = luma_dev; cp.H = H; cp.W = W; cp.stride = (size_t)stride;
        cp.f_begin = f; cp.n_frames = n_frames; cp.max_frames = (chain_run<RELAY_AFTER) ? (RELAY_AFTER-chain_run) : CHAIN_LAUNCH_FRAMES;
        const int f_launch = f;
        cp.recs = recs_dev; cp.aux = aux_dev; cp.ctx = h->ctx;
        cp.clean = h->clean; cp.have_spec = have_spec ? 1 : 0; cp.spec_ref = spec_ref; cp.spec_coords = spec_c;
        cp.reset = ((f==0)&&!cont) ? 1 : 0; cp.mode = cfg->mode; cp.line_dup = dup_flags; cp.segments = 1; cp.cont = cont ? 1 : 0;
        stc007_chain_kernel<1024><<<1, 1024, 0, st>>>(cp);
        h->stats.kernel_launches++;
        { int rc = read_hdr(h, st); if(rc) return rc; }
        f = h->hdr_host->next_frame;
        bool warm_hit = false;
        if(warm_pending)
        {   // join the speculative bulk launch
            warm_pending = false;
            const BinState &wb = h->warm_bin, &cb = h->hdr_host->bin;
            warm_hit = (f==1)&&h->hdr_host->stable&&(wb.def_ref==cb.def_ref)&&coord_eq(wb.def_coord, cb.def_coord)
                       &&(wb.def_black==cb.def_black)&&(wb.def_white==cb.def_white);
            if(warm_hit&&h->first_frame_fn&&!h->first_frame_called)
            {   // frame 0's records are final and the bulk pass is still running on its own stream: the caller's chance to
                // start work that needs only them (the halo for the previous shard) -- before [st] is joined to that pass
                h->first_frame_called = 1;
                h->first_frame_fn(h->first_frame_user);
            }
            CK(cudaStreamWaitEvent(st, h->ev_sync[1], 0));
            if(!warm_hit)
            {   // wrong guess: its records may have raced with the chain kernel's; start over without it
                CK(cudaStreamSynchronize(st));
                h->warm_valid = 0;
                if(fuse_req) h->fuse_arm.armed = 1;
                return decode_frames_impl(h, cfg, luma_dev, n_frames, H, W, stride, recs_dev, aux_dev, cuda_stream);
            }
            have_spec = true; spec_ref = wb.def_ref; spec_c = wb.def_coord; spec_black = wb.def_black; spec_white = wb.def_white;
        }
        if(f>=n_frames) break;
        if(!h->hdr_host->stable)
        {
            // A whole launch of frames without the chain settling: a damaged tape.  The rest is decoded in relay mode --
            // many chains at once, each verified to have started from the true state (see relay_decode).
            chain_run += f-f_launch;
            continue;
        }
        chain_run += f-f_launch;
        const BinState b = h->hdr_host->bin;
        bool bulk_ran = warm_hit;
        if(!have_spec||(spec_ref!=b.def_ref)||!coord_eq(spec_c, b.def_coord))
        {
            launch_bulk(st, f, b, &h->ctx->first_unclean);
            have_spec = true; spec_ref = b.def_ref; spec_c = b.def_coord; spec_black = b.def_black; spec_white = b.def_white;
            bulk_ran = true;        // the bulk kernel left the first frame it could not take in ctx->first_unclean
        }
        if(!bulk_ran)
        {
            first_unclean_kernel<<<1, 1024, 0, st>>>(h->clean, f, n_frames, h->ctx);
            h->stats.kernel_launches++;
        }
        int fb;
        if(warm_hit&&(cfg->reserved[2]&2)&&!cont)
        {
            // Lazy verification: do not wait for the bulk pass to learn that it took every frame (it nearly always does).  Everything
            // the success case still has to do is enqueued with the count read on the device; the call returns, the caller goes
            // on enqueuing what follows, and sdv_bin_decode_verify() looks at the answer later -- and decodes the tape again,
            // without speculation, in the rare case that a frame was not clean.
            if((b.def_black!=spec_black)||(b.def_white!=spec_white))
            {
                const size_t cnt = (size_t)(n_frames-f)*H;
                patch_bw_kernel<<<(unsigned)((cnt+255)/256), 256, 0, st>>>(recs_dev, (size_t)f*H, cnt, b.def_black, b.def_white);
                h->stats.kernel_launches++;
            }
            chain_skip_dev_kernel<<<1, 1, 0, st>>>(h->ctx, h->spec_fu, f);
            h->stats.kernel_launches++;
            CK(cudaMemcpyAsync(h->fu_host, h->spec_fu, sizeof(int), cudaMemcpyDeviceToHost, st));
            CK(cudaEventRecord(h->ev_lazy, st));
            h->lazy_pending = 1; h->lazy_cfg = *cfg; h->lazy_luma = luma_dev; h->lazy_n = n_frames; h->lazy_H = H; h->lazy_W = W; h->lazy_stride = stride;
            h->lazy_recs = recs_dev; h->lazy_aux = aux_dev; h->lazy_stream = cuda_stream;
            frames_bulk += (uint64_t)(n_frames-f);
            f = n_frames;
            break;
        }
        if(warm_hit)
        {
            CK(cudaMemcpyAsync(h->fu_host, h->spec_fu, sizeof(int), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            fb = *h->fu_host;
        }
        else
        {
            { int rc = read_hdr(h, st); if(rc) return rc; }
            fb = h->hdr_host->first_unclean;
        }
        if(fb<n_frames) fuse_ok = false;            // a frame the bulk pass could not take: its fused blocks are void
        if(fb>f)
        {
            if((b.def_black!=spec_black)||(b.def_white!=spec_white))
            {
                const size_t cnt = (size_t)(fb-f)*H;
                patch_bw_kernel<<<(unsigned)((cnt+255)/256), 256, 0, st>>>(recs_dev, (size_t)f*H, cnt, b.def_black, b.def_white);
                h->stats.kernel_launches++;
            }
            {   // the chain continues after the clean run (in this call, or in the call that continues the file): account for
                // the frames it did not see
                chain_skip_kernel<<<1, 1, 0, st>>>(h->ctx, fb-f);
                h->stats.kernel_launches++;
            }
            frames_bulk += (uint64_t)(fb-f);
            f = fb;
            chain_run = 0;
        }
    }
    CK(cudaGetLastError());
    if(have_spec)
    {   // remember the steady-state presets for the next call's warm start
        h->warm_valid = 1; h->warm_H = H; h->warm_W = W; h->warm_mode = cfg->mode|(dup_flags<<8);
        h->warm_bin = BinState(); h->warm_bin.def_ref = spec_ref; h->warm_bin.def_coord = spec_c;
        h->warm_bin.def_black = spec_black; h->warm_bin.def_white = spec_white;
    }
    h->chain_open = 1; h->chain_H = H; h->chain_W = W; h->chain_mode = cfg->mode|(dup_flags<<8);
    if(fuse_req&&fuse_ok&&(fuse_launches==1)&&(frames_bulk==(uint64_t)(n_frames-fuse_from)))
    {
        h->fuse_done.valid = 1; h->fuse_done.n_frames = n_frames; h->fuse_done.H = H; h->fuse_done.f_from = fuse_from;
        h->fuse_done.lead_in = h->fuse_arm.geo.lead_in; h->fuse_done.lpf = h->fuse_arm.geo.lines_per_field; h->fuse_done.dur = h->fuse_arm.cfg.broken_mask_dur;
        h->fuse_done.samples = h->fuse_arm.samples; h->fuse_done.sflags = h->fuse_arm.sflags; h->fuse_done.recs = recs_dev;
    }
    h->stats.lines_fast = frames_bulk*(uint64_t)H;
    h->stats.lines_chain = h->stats.lines_total-h->stats.lines_fast;
    h->stats.frames_skipped = frames_bulk;
    if(!relayed) h->stats.reserved = (uint32_t)h->hdr_host->lines_swept;
    h->acc_launches += h->stats.kernel_launches;
    return SDV_OK;
}

int sdv_bin_decode_verify(sdv_handle *h, int *redone)
{
    if(!h) return SDV_ERR_ARG;
    if(redone) *redone = 0;
    if(!h->lazy_pending) return SDV_OK;
    CK(cudaSetDevice(h->device));
    CK(cudaEventSynchronize(h->ev_lazy));
    h->lazy_pending = 0;
    if(*h->fu_host>=h->lazy_n) return SDV_OK;
    // a frame the bulk pass could not take: the speculation does not stand, the tape is decoded again the ordinary way
    sdv_bin_config c = h->lazy_cfg;
    c.reserved[2] = (uint8_t)((c.reserved[2]&~2)|1);
    h->warm_valid = 0;
    const int rc = decode_frames_impl(h, &c, h->lazy_luma, h->lazy_n, h->lazy_H, h->lazy_W, h->lazy_stride, h->lazy_recs, h->lazy_aux, h->lazy_stream);
    if(rc) return rc;
    if(redone) *redone = 1;
    return SDV_OK;
}

// ---- the open file of the line decode as a blob (layout: CS_* in chain_state.cuh)
static_assert(sizeof(sdv_bin_preset)==32, "blob layout of the fine settings");

int sdv_bin_chain_state_bytes(void) { return CS_BYTES; }

int sdv_bin_chain_state_save(sdv_handle *h, int pcm_type, void *state_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!state_dev||((uintptr_t)state_dev%4)) return fail(h, SDV_ERR_ARG, "sdv_bin_chain_state_save: null or misaligned state buffer", cudaSuccess);
    if(h->lazy_pending) return fail(h, SDV_ERR_ARG, "sdv_bin_chain_state_save: the previous call was lazy (reserved[2] bit 1): call sdv_bin_decode_verify first", cudaSuccess);
    int kind, H, W, mode, dup;
    const void *ctx;
    if((pcm_type==SDV_TYPE_STC007)||(pcm_type==SDV_TYPE_M2))
    {
        if(!h->chain_open||(((h->chain_mode>>9)&1)!=((pcm_type==SDV_TYPE_M2) ? 1 : 0)))
            return fail(h, SDV_ERR_ARG, "sdv_bin_chain_state_save: no open file of this PCM type on the handle", cudaSuccess);
        kind = CS_KIND_STC; ctx = h->ctx; H = h->chain_H; W = h->chain_W; mode = h->chain_mode&0xFF; dup = (h->chain_mode>>8)&1;
    }
    else if((pcm_type==SDV_TYPE_PCM1)||(pcm_type==SDV_TYPE_PCM16X0))
    {
        if(!h->pcm_open||(h->pcm_type!=pcm_type))
            return fail(h, SDV_ERR_ARG, "sdv_bin_chain_state_save: no open file of this PCM type on the handle", cudaSuccess);
        kind = (pcm_type==SDV_TYPE_PCM1) ? CS_KIND_P1 : CS_KIND_X0; ctx = (kind==CS_KIND_P1) ? (const void *)h->p1_ctx : (const void *)h->x0_ctx;
        H = h->pcm_H; W = h->pcm_W; mode = h->pcm_mode&0xFF; dup = (h->pcm_mode>>8)&1;
    }
    else return fail(h, SDV_ERR_ARG, "sdv_bin_chain_state_save: pcm_type", cudaSuccess);
    CK(cudaSetDevice(h->device));
    ChainBlobHdr hdr; memset(&hdr, 0, sizeof(hdr));
    u8 *b = (u8 *)hdr.w;
    cs_put32(b, CSH_MAGIC, CS_MAGIC); cs_put16(b, CSH_VERSION, CS_VERSION); cs_put16(b, CSH_TYPE, (u32)pcm_type); cs_put32(b, CSH_SIZE, CS_BYTES);
    cs_put16(b, CSH_H, (u32)H); cs_put16(b, CSH_W, (u32)W); b[CSH_MODE] = (u8)mode; b[CSH_DUP] = (u8)dup; b[CSH_M2] = (pcm_type==SDV_TYPE_M2) ? 1 : 0;
    sdv_bin_preset fine; sdv_bin_get_fine_settings(h, &fine);
    memcpy(b+CSH_FINE, &fine, sizeof(fine));
    chain_state_pack_kernel<<<1, 128, 0, (cudaStream_t)cuda_stream>>>(hdr, kind, ctx, (u32 *)state_dev);
    h->acc_launches += 1;
    CK(cudaGetLastError());
    return SDV_OK;
}

int sdv_bin_chain_state_load(sdv_handle *h, const void *state_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!state_dev||((uintptr_t)state_dev%4)) return fail(h, SDV_ERR_ARG, "sdv_bin_chain_state_load: null or misaligned state buffer", cudaSuccess);
    if(h->lazy_pending) return fail(h, SDV_ERR_ARG, "sdv_bin_chain_state_load: the previous call was lazy (reserved[2] bit 1): call sdv_bin_decode_verify first", cudaSuccess);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    std::vector<u8> blob(CS_BYTES);
    CK(cudaMemcpyAsync(blob.data(), state_dev, CS_BYTES, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const u8 *b = blob.data();
    const int kind = cs_blob_kind(b);
    if(kind<0) return fail(h, SDV_ERR_ARG, "sdv_bin_chain_state_load: not a line-decode chain state of this version", cudaSuccess);
    {   // canonical: the state it holds packs to the same bytes (history entries past the counts and unused bytes zero)
        std::vector<u8> again(blob.begin(), blob.begin()+CS_HDR);
        again.resize(CS_BYTES, 0);
        if(kind==CS_KIND_STC) { std::unique_ptr<ChainCtx> x(new ChainCtx()); cs_unpack_stc(b, x.get()); cs_pack_stc(x.get(), again.data()); }
        else if(kind==CS_KIND_P1) { std::unique_ptr<P1ChainCtx> x(new P1ChainCtx()); cs_unpack_p1(b, x.get()); cs_pack_p1(x.get(), again.data()); }
        else { std::unique_ptr<X0ChainCtx> x(new X0ChainCtx()); cs_unpack_x0(b, x.get()); cs_pack_x0(x.get(), again.data()); }
        if(memcmp(again.data(), b, CS_BYTES)) return fail(h, SDV_ERR_ARG, "sdv_bin_chain_state_load: the blob is not in canonical form", cudaSuccess);
    }
    sdv_bin_preset fine; sdv_bin_get_fine_settings(h, &fine);
    if(memcmp(b+CSH_FINE, &fine, sizeof(fine)))
        return fail(h, SDV_ERR_ARG, "sdv_bin_chain_state_load: the handle's fine settings differ from the ones the state was saved with", cudaSuccess);
    const int type = (int)cs_get16(b, CSH_TYPE), H = (int)cs_get16(b, CSH_H), W = (int)cs_get16(b, CSH_W);
    const int key_mode = (int)b[CSH_MODE]|((int)b[CSH_DUP]<<8);
    void *ctx = (kind==CS_KIND_STC) ? (void *)h->ctx : ((kind==CS_KIND_P1) ? (void *)h->p1_ctx : (void *)h->x0_ctx);
    if(kind==CS_KIND_STC) h->chain_open = 0; else h->pcm_open = 0;
    if(kind==CS_KIND_STC) chain_state_unpack_kernel<CS_KIND_STC><<<1, 128, 0, st>>>((const u32 *)state_dev, ctx);
    else if(kind==CS_KIND_P1) chain_state_unpack_kernel<CS_KIND_P1><<<1, 128, 0, st>>>((const u32 *)state_dev, ctx);
    else chain_state_unpack_kernel<CS_KIND_X0><<<1, 128, 0, st>>>((const u32 *)state_dev, ctx);
    h->acc_launches += 1;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    if(kind==CS_KIND_STC) { h->chain_open = 1; h->chain_H = H; h->chain_W = W; h->chain_mode = key_mode|((int)b[CSH_M2]<<9); }
    else { h->pcm_open = 1; h->pcm_type = type; h->pcm_H = H; h->pcm_W = W; h->pcm_mode = key_mode; }
    return SDV_OK;
}

int sdv_timings_read(sdv_handle *h, sdv_timings *out, int reset)
{
    if(!h||!out) return SDV_ERR_ARG;
    memset(out, 0, sizeof(*out));
    CK(cudaSetDevice(h->device));
    timing_flush(h, 0); timing_flush(h, 1);
    out->bulk_ms = (float)h->acc_ms[0]; out->bulk_lines = h->acc_units[0]; out->bulk_launches = h->acc_n[0];
    out->deint_ms = (float)h->acc_ms[1]; out->deint_blocks = h->acc_units[1]; out->deint_launches = h->acc_n[1];
    out->kernel_launches = h->acc_launches;
    if(reset) { h->acc_ms[0] = h->acc_ms[1] = 0; h->acc_units[0] = h->acc_units[1] = 0; h->acc_n[0] = h->acc_n[1] = 0; h->acc_launches = 0; }
    return SDV_OK;
}

int sdv_bin_last_stats(sdv_handle *h, sdv_bin_stats *out)
{
    if(!h||!out) return SDV_ERR_ARG;
    *out = h->stats;
    return SDV_OK;
}

// Scratch of one deinterleave pass: candidate bits, their summary bytes, the window list.
static DeintCfg make_deint_cfg(const sdv_deint_config *cfg)
{
    DeintCfg c;
    c.res_mode = cfg->res_mode; c.ignore_crc = cfg->ignore_crc; c.force_check = cfg->force_check;
    c.q_corr = cfg->q_corr ? 1 : 0; c.m2 = cfg->m2_format ? 1 : 0;
    c.p_corr = (cfg->p_corr||cfg->q_corr) ? 1 : 0;          // setQCorrection(true) implies setPCorrection(true) (stc007deinterleaver.cpp:210-260)
    return c;
}
__global__ void set_countdown_kernel(int *state, int v) { state[0] = v; state[1] = 0; state[2] = 0; state[3] = 0; }

// The countdown windows after a first pass (stream ordered, no host round trip): walk the candidates, redo the blocks
// inside windows.  [countdown_in]: what the blocks before this stream left of an open window.
static int run_windows(sdv_handle *h, const DeintScratch &sc, WindowParams &wp, int dur, int countdown_in, cudaStream_t st)
{
    broken_window_kernel<<<1, 1024, 0, st>>>(sc.bits, sc.sum, wp.n_blocks, dur, countdown_in, sc.wl);
    wp.wl = sc.wl;
    stc007_window_kernel<<<2*h->num_sms, 128, 0, st>>>(wp);
    h->acc_launches += 2;
    return SDV_OK;
}

// stc007_deint_kernel<true> wherever it applies: the standard setting without the M2 expansion, no block records, both output
// buffers aligned for the 8-byte sample / 4-byte flag stores of a pair, and every tile starting on an even block.
static bool deint_pair_applies(const DeintParams &p)
{
    return deint_cfg_is_std14(p.cfg)&&(!p.cfg.m2)&&(!p.blocks)&&p.samples&&p.sflags&&((((uintptr_t)p.samples)&7u)==0)
           &&((((uintptr_t)p.sflags)&3u)==0)&&((p.tile_base&1)==0)&&((p.tile_stride&1)==0);
}
static void launch_deint(const DeintParams &p, unsigned grid, cudaStream_t st)
{
    if(deint_pair_applies(p)) stc007_deint_kernel<true><<<grid, DEINT_THREADS, 0, st>>>(p);
    else stc007_deint_kernel<false><<<grid, DEINT_THREADS, 0, st>>>(p);
}

static int run_deint(sdv_handle *h, const sdv_deint_config *cfg, const AsmMap &map, long long n_blocks,
                     sdv_block_rec *blocks_dev, int16_t *samples_dev, uint8_t *sample_flags_dev, cudaStream_t st)
{
    if(n_blocks<=0) return SDV_OK;
    if(cfg->cwd) return fail(h, SDV_ERR_UNSUPPORTED, "CWD needs the stitcher's frame queue: use sdv_stc007_stitch_frames (sdv_deint_config.cwd)", cudaSuccess);
    DeintScratch sc;
    { int rc = deint_scratch(h, n_blocks, cfg->broken_mask_dur, &sc); if(rc) return rc; }
    DeintParams p;
    p.map = map; p.n_blocks = n_blocks;
    p.cfg = make_deint_cfg(cfg);
    p.blocks = blocks_dev; p.samples = samples_dev; p.sflags = sample_flags_dev;
    const bool windows = cfg->broken_mask_dur>0;
    p.broken_bits = windows ? sc.bits : NULL; p.broken_sum = windows ? sc.sum : NULL;
    p.tile_base = 0; p.tile_stride = DEINT_TILE; p.tile_len = DEINT_TILE; p.atomic_bits = 0;
    p.n_tiles = (int)((n_blocks+DEINT_TILE-1)/DEINT_TILE);
    // Did the decode call that produced these records also finish the blocks that lie inside a frame (fused bulk pass)?  Then only
    // the rest is left: everything in front of the first fused frame, and the last 112 blocks of every frame.
    const auto &fd = h->fuse_done;
    const bool fused = fd.valid&&map.geo&&(!blocks_dev)&&(samples_dev==fd.samples)&&(sample_flags_dev==fd.sflags)&&(map.recs==fd.recs)
                       &&(map.lead_in==fd.lead_in)&&(map.lpf==fd.lpf)&&(map.H==fd.H)&&(map.n_fields==2*(long long)fd.n_frames)&&(cfg->broken_mask_dur==fd.dur)
                       &&deint_cfg_is_std14(p.cfg)&&(!p.cfg.ignore_crc)&&(!p.cfg.m2)&&windows;
    h->fuse_done.valid = 0;
    timing_flush(h, 1);
    cudaEventRecord(h->ev[2], st);
    if(fused)
    {
        p.atomic_bits = 1;
        const long long head = (long long)fd.lead_in+(long long)fd.f_from*2*fd.lpf;       // blocks in front of the first fused frame
        if(head>0)
        {
            DeintParams q = p;
            q.n_blocks = (head<n_blocks) ? head : n_blocks;
            q.n_tiles = (int)((q.n_blocks+DEINT_TILE-1)/DEINT_TILE);
            launch_deint(q, (unsigned)((q.n_tiles+DEINT_WARPS-1)/DEINT_WARPS), st);
            h->acc_launches += 1;
        }
        const int n_rest = fd.n_frames-fd.f_from;
        if(n_rest>0)
        {
            DeintParams q = p;
            q.tile_base = head+(2*fd.lpf-112); q.tile_stride = 2*fd.lpf; q.tile_len = 112; q.n_tiles = n_rest;
            launch_deint(q, (unsigned)((q.n_tiles+DEINT_WARPS-1)/DEINT_WARPS), st);
            h->acc_launches += 1;
        }
    }
    else
    {
        if(windows) CK(cudaMemsetAsync(sc.sum, 0, (size_t)((n_blocks+1023)>>10), st));
        const unsigned grid = (unsigned)((n_blocks+DEINT_CTA_BLOCKS-1)/DEINT_CTA_BLOCKS);
        launch_deint(p, grid, st);
        h->acc_launches += 1;
    }
    cudaEventRecord(h->ev[3], st);
    h->ev_set[1] = 1; h->ev_units[1] = (uint64_t)n_blocks;
    if(windows)
    {
        WindowParams wp; memset(&wp, 0, sizeof(wp));
        wp.stitched = 0; wp.amap = map; wp.n_blocks = n_blocks; wp.cfg = p.cfg;
        wp.blocks = blocks_dev; wp.samples = samples_dev; wp.sflags = sample_flags_dev;
        int rc = run_windows(h, sc, wp, cfg->broken_mask_dur, cfg->countdown_in, st);
        if(rc) return rc;
    }
    CK(cudaGetLastError());
    return SDV_OK;
}

int sdv_stc007_fuse_next_decode(sdv_handle *h, const sdv_deint_config *cfg, const sdv_stc007_geometry *geo, int16_t *samples_dev, uint8_t *sample_flags_dev)
{
    if(!h) return SDV_ERR_ARG;
    h->fuse_arm.armed = 0;
    if(!cfg||!geo||!samples_dev||!sample_flags_dev||((uintptr_t)samples_dev%4)||((uintptr_t)sample_flags_dev%2))
        return fail(h, SDV_ERR_ARG, "sdv_stc007_fuse_next_decode: null or misaligned buffers", cudaSuccess);
    const DeintCfg c = make_deint_cfg(cfg);
    if(!deint_cfg_is_std14(c)||c.ignore_crc||c.m2||cfg->cwd||(cfg->broken_mask_dur==0)||(geo->lines_per_field<120))
        return SDV_OK;          // not the standard setting: nothing is fused, the deinterleave call does all the work
    h->fuse_arm.armed = 1; h->fuse_arm.cfg = *cfg; h->fuse_arm.geo = *geo; h->fuse_arm.samples = samples_dev; h->fuse_arm.sflags = sample_flags_dev;
    return SDV_OK;
}

int sdv_stc007_countdown_copy(sdv_handle *h, int32_t *state_dev, void *cuda_stream)
{
    if(!h||!state_dev) return SDV_ERR_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(state_dev, h->win_state, 4*sizeof(int), cudaMemcpyDeviceToDevice, (cudaStream_t)cuda_stream));
    return SDV_OK;
}

int sdv_stc007_countdown(sdv_handle *h, sdv_countdown *out, void *cuda_stream)
{
    if(!h||!out) return SDV_ERR_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    CK(cudaMemcpyAsync(h->win_state_host, h->win_state, 4*sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    out->countdown_in = (uint8_t)h->win_state_host[0]; out->countdown_out = (uint8_t)h->win_state_host[1];
    out->depends_on_in = (uint8_t)h->win_state_host[3]; out->reserved = 0; out->windows = (uint32_t)h->win_state_host[2];
    return SDV_OK;
}

int sdv_deint_stc007(sdv_handle *h, const sdv_deint_config *cfg, const sdv_line_rec *asm_lines_dev, int n_lines,
                     sdv_block_rec *blocks_dev, int16_t *samples_dev, uint8_t *sample_flags_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!cfg||(n_lines<0)||(cfg->res_mode>SDV_RES_MODE_16BIT)) return fail(h, SDV_ERR_ARG, "sdv_deint_stc007", cudaSuccess);
    if(n_lines<=112) return SDV_OK;         // DI_RET_NO_DATA: not enough lines for one block
    if(!asm_lines_dev||((uintptr_t)asm_lines_dev%16)) return fail(h, SDV_ERR_ARG, "sdv_deint_stc007: null or misaligned lines", cudaSuccess);
    CK(cudaSetDevice(h->device));
    AsmMap m; memset(&m, 0, sizeof(m));
    m.recs = asm_lines_dev; m.n_lines = n_lines; m.geo = 0;
    return run_deint(h, cfg, m, (long long)n_lines-112, blocks_dev, samples_dev, sample_flags_dev, (cudaStream_t)cuda_stream);
}

int sdv_deint_pcm1(sdv_handle *h, int ignore_crc, const sdv_pcm1_subline *sublines_dev, int n_fields,
                   int16_t *samples_dev, uint8_t *sample_flags_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if((n_fields<0)||(n_fields>(1<<24))) return fail(h, SDV_ERR_ARG, "sdv_deint_pcm1", cudaSuccess);
    if(n_fields==0) return SDV_OK;
    if(!sublines_dev||!samples_dev||((uintptr_t)sublines_dev%8)||((uintptr_t)samples_dev%2))
        return fail(h, SDV_ERR_ARG, "sdv_deint_pcm1: null or misaligned buffer", cudaSuccess);
    CK(cudaSetDevice(h->device));
    pcm1_deint_kernel<<<(unsigned)n_fields*P1_BLOCKS, P1_THREADS, 0, (cudaStream_t)cuda_stream>>>(sublines_dev, n_fields, ignore_crc, samples_dev, sample_flags_dev);
    h->acc_launches += 1;
    CK(cudaGetLastError());
    return SDV_OK;
}

int sdv_pcm1_frames_to_samples(sdv_handle *h, const sdv_pcm1_stitch_config *cfg, const sdv_line_rec *recs_dev, int n_frames, int H,
                               int16_t *samples_dev, uint8_t *sample_flags_dev, sdv_pcm1_frame_info *info_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!cfg) return fail(h, SDV_ERR_ARG, "sdv_pcm1_frames_to_samples", cudaSuccess);
    const int ignore_crc = cfg->ignore_crc, bff = cfg->bff, file_start = cfg->file_start;
    if((n_frames<0)||(n_frames>(1<<23))||(H<2)||(H&1)||(H>2*SDV_MAX_H)) return fail(h, SDV_ERR_ARG, "sdv_pcm1_frames_to_samples", cudaSuccess);
    if(n_frames==0) return SDV_OK;
    if(!recs_dev||!samples_dev||((uintptr_t)recs_dev%16)||((uintptr_t)samples_dev%2)||((uintptr_t)info_dev%2))
        return fail(h, SDV_ERR_ARG, "sdv_pcm1_frames_to_samples: null or misaligned buffer", cudaSuccess);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    { int rc = ensure(h, (void **)&h->p1_sub, &h->p1_sub_cap, (size_t)n_frames*2*P1S_SUBLINES_PF*sizeof(sdv_pcm1_subline)); if(rc) return rc; }
    pcm1_assemble_kernel<<<n_frames, 256, 0, st>>>(recs_dev, n_frames, H, bff, file_start, cfg->manual_offset, cfg->odd_offset, cfg->even_offset,
                                                   h->p1_sub, info_dev);
    timing_flush(h, 1);
    cudaEventRecord(h->ev[2], st);
    pcm1_deint_kernel<<<(unsigned)n_frames*2*P1_BLOCKS, P1_THREADS, 0, st>>>(h->p1_sub, n_frames*2, ignore_crc, samples_dev, sample_flags_dev);
    cudaEventRecord(h->ev[3], st);
    h->ev_set[1] = 1; h->ev_units[1] = (uint64_t)n_frames*2*P1_BLOCKS;
    h->acc_launches += 2;
    CK(cudaGetLastError());
    return SDV_OK;
}

int sdv_pcm16x0_frames_to_samples(sdv_handle *h, const sdv_pcm16x0_config *cfg, const sdv_pcm16x0_geometry *geo, const sdv_line_rec *recs_dev,
                                  int n_frames, int H, const uint8_t *mask_seams_dev, int16_t *samples_dev, uint8_t *sample_flags_dev,
                                  void *cuda_stream)
{
    return sdv_pcm16x0_frames_to_samples_info(h, cfg, geo, recs_dev, n_frames, H, mask_seams_dev, samples_dev, sample_flags_dev, NULL, cuda_stream);
}

// The control-bit history of the PCM-16x0 stitch calls: every call leaves the votes of its file's last X0_CTRL_HISTORY frames in
// one of the handle's two vote buffers; a call with continue_file votes with what the call before left, otherwise with none.
static int x0_votes_begin(sdv_handle *h, const sdv_pcm16x0_config *cfg, int ei, const u8 **hist_in, u8 **hist_out)
{
    if(cfg->continue_file&&(h->x0_votes_open!=1+ei))
        return fail(h, SDV_ERR_ARG, "PCM-16x0 stitcher: nothing to continue (continue_file without an earlier stitch call in this format on the handle)", cudaSuccess);
    *hist_in = cfg->continue_file ? h->x0_votes+h->x0_votes_cur*X0_CTRL_HISTORY : NULL;
    *hist_out = h->x0_votes+(1-h->x0_votes_cur)*X0_CTRL_HISTORY;
    h->x0_votes_open = 0;
    return SDV_OK;
}
static void x0_votes_end(sdv_handle *h, int ei) { h->x0_votes_cur = 1-h->x0_votes_cur; h->x0_votes_open = 1+ei; }

int sdv_pcm16x0_frames_to_samples_info(sdv_handle *h, const sdv_pcm16x0_config *cfg, const sdv_pcm16x0_geometry *geo, const sdv_line_rec *recs_dev,
                                       int n_frames, int H, const uint8_t *mask_seams_dev, int16_t *samples_dev, uint8_t *sample_flags_dev,
                                       sdv_pcm16x0_frame_info *info_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!cfg||!geo||(n_frames<0)||(n_frames>(1<<23))||(H<2)||(H&1)||(H>2*SDV_MAX_H)||(geo->top_padding_odd>X0S_LINES_PF)||(geo->top_padding_even>X0S_LINES_PF))
        return fail(h, SDV_ERR_ARG, "sdv_pcm16x0_frames_to_samples", cudaSuccess);
    if(n_frames==0) return SDV_OK;
    if(!recs_dev||!samples_dev||((uintptr_t)recs_dev%16)||((uintptr_t)samples_dev%2))
        return fail(h, SDV_ERR_ARG, "sdv_pcm16x0_frames_to_samples: null or misaligned buffer", cudaSuccess);
    const int ei = cfg->ei_format ? 1 : 0;
    const u8 *hist_in = NULL; u8 *hist_out = NULL;
    { const int rc = x0_votes_begin(h, cfg, ei, &hist_in, &hist_out); if(rc) return rc; }
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    X0Cfg c; c.ignore_crc = cfg->ignore_crc; c.force_check = cfg->force_check; c.p_corr = cfg->p_corr;
    timing_flush(h, 1);
    cudaEventRecord(h->ev[2], st);
    pcm16x0_stitch_kernel<<<n_frames, 512, 0, st>>>(recs_dev, n_frames, H, geo->bff, geo->top_padding_odd, geo->top_padding_even, c,
                                                    geo->broken_mask_dur, mask_seams_dev, samples_dev, sample_flags_dev, info_dev, ei, hist_in, hist_out);
    cudaEventRecord(h->ev[3], st);
    h->ev_set[1] = 1; h->ev_units[1] = (uint64_t)n_frames*X0S_BLOCKS_FRAME;
    h->acc_launches += 1;
    if(info_dev)
    {
        if((uintptr_t)info_dev%2) return fail(h, SDV_ERR_ARG, "sdv_pcm16x0_frames_to_samples_info: misaligned info", cudaSuccess);
        pcm16x0_ctrl_history_kernel<<<(unsigned)((n_frames+255)/256), 256, 0, st>>>(info_dev, n_frames, hist_in);
        h->acc_launches += 1;
    }
    CK(cudaGetLastError());
    x0_votes_end(h, ei);
    return SDV_OK;
}

int sdv_pcm16x0_frames_to_samples_auto(sdv_handle *h, const sdv_pcm16x0_config *cfg, const sdv_pcm16x0_geometry *geo, const sdv_line_rec *recs_dev,
                                       int n_frames, int H, int file_start, int mask_seams, int16_t *samples_dev, uint8_t *sample_flags_dev,
                                       sdv_pcm16x0_frame_info *info_dev, sdv_pcm16x0_alignment *align_host, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!cfg||!geo||(n_frames<0)||(n_frames>(1<<23))||(H<2)||(H&1)||(H>2*SDV_MAX_H)) return fail(h, SDV_ERR_ARG, "sdv_pcm16x0_frames_to_samples_auto", cudaSuccess);
    if(n_frames==0) return SDV_OK;
    if(!recs_dev||!samples_dev||((uintptr_t)recs_dev%16)||((uintptr_t)samples_dev%2)||((uintptr_t)info_dev%2))
        return fail(h, SDV_ERR_ARG, "sdv_pcm16x0_frames_to_samples_auto: null or misaligned buffer", cudaSuccess);
    if(cfg->continue_file&&file_start)
        return fail(h, SDV_ERR_ARG, "sdv_pcm16x0_frames_to_samples_auto: continue_file with file_start (a call either opens the file or continues it)", cudaSuccess);
    const int ei = cfg->ei_format ? 1 : 0;
    const u8 *hist_in = NULL; u8 *hist_out = NULL;
    int rc;
    if((rc = x0_votes_begin(h, cfg, ei, &hist_in, &hist_out))) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if((rc = ensure(h, (void **)&h->x0_scan, &h->x0_scan_cap, 2*(size_t)n_frames*sizeof(X0PadScan)))) return rc;
    if((rc = ensure(h, (void **)&h->x0_geo, &h->x0_geo_cap, 2*(size_t)n_frames*sizeof(X0FieldGeo)))) return rc;
    if((rc = ensure(h, (void **)&h->x0_mask, &h->x0_mask_cap, (size_t)n_frames+16))) return rc;
    X0Cfg c; c.ignore_crc = cfg->ignore_crc; c.force_check = cfg->force_check; c.p_corr = cfg->p_corr;
    // a change of format drops the padding history (PCM16X0DataStitcher::setFormat -> resetState, 5456-5490, 5671-5676)
    if(file_start||(h->x0_pads_open!=1+ei)) h->x0_pads.reset();
    h->x0_pads.p_corr = cfg->p_corr!=0;
    h->x0_pads_open = 1+ei;
    std::vector<X0FieldGeo> fg(2*(size_t)n_frames);
    std::vector<u8> mask((size_t)n_frames);
    std::vector<X0PadScan> scan;
    std::vector<X0EIScan> scan_ei;
    if(ei)
    {   // per frame: tryEIPadding x 81 paddings between the fields, control-bit offsets from the bottom of either field
        if((rc = ensure(h, (void **)&h->x0_scan_ei, &h->x0_scan_ei_cap, (size_t)n_frames*sizeof(X0EIScan)))) return rc;
        pcm16x0_eipad_kernel<<<(unsigned)n_frames, 256, 0, st>>>(recs_dev, n_frames, H, geo->bff, c, h->x0_scan_ei);
        scan_ei.resize((size_t)n_frames);
        CK(cudaMemcpyAsync(scan_ei.data(), h->x0_scan_ei, scan_ei.size()*sizeof(X0EIScan), cudaMemcpyDeviceToHost, st));
    }
    else
    {   // per field: trySIPadding x 35 paddings, control-bit offset, interleave block estimate
        pcm16x0_sipad_kernel<<<2*(unsigned)n_frames, 256, 0, st>>>(recs_dev, n_frames, H, c, h->x0_scan);
        scan.resize(2*(size_t)n_frames);
        CK(cudaMemcpyAsync(scan.data(), h->x0_scan, scan.size()*sizeof(X0PadScan), cudaMemcpyDeviceToHost, st));
    }
    h->acc_launches += 1;
    CK(cudaStreamSynchronize(st));
    // the decisions, frame by frame (the padding history makes them sequential)
    for(int f=0;f<n_frames;f++)
    {
        uint8_t res[2];
        const bool m = ei ? h->x0_pads.frame_ei(scan_ei[(size_t)f], geo->bff!=0, &fg[2*(size_t)f], res)
                          : h->x0_pads.frame(scan[2*(size_t)f], scan[2*(size_t)f+1], &fg[2*(size_t)f], res);
        mask[f] = (m&&mask_seams) ? 1 : 0;
        if(align_host)
        {
            sdv_pcm16x0_alignment a; memset(&a, 0, sizeof(a));
            for(int k=0;k<2;k++) { a.top_padding[k] = fg[2*(size_t)f+k].top_pad; a.cut_lines[k] = fg[2*(size_t)f+k].cut; a.lines[k] = fg[2*(size_t)f+k].lines; a.result[k] = res[k]; }
            a.mask_seams = mask[f];
            align_host[f] = a;
        }
    }
    CK(cudaMemcpyAsync(h->x0_geo, fg.data(), fg.size()*sizeof(X0FieldGeo), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->x0_mask, mask.data(), mask.size(), cudaMemcpyHostToDevice, st));
    timing_flush(h, 1);
    cudaEventRecord(h->ev[2], st);
    pcm16x0_stitch_geo_kernel<<<n_frames, 512, 0, st>>>(recs_dev, n_frames, H, geo->bff, h->x0_geo, c, geo->broken_mask_dur, h->x0_mask,
                                                        samples_dev, sample_flags_dev, info_dev, ei, hist_in, hist_out);
    cudaEventRecord(h->ev[3], st);
    h->ev_set[1] = 1; h->ev_units[1] = (uint64_t)n_frames*X0S_BLOCKS_FRAME;
    h->acc_launches += 1;
    if(info_dev)
    {
        pcm16x0_ctrl_history_kernel<<<(unsigned)((n_frames+255)/256), 256, 0, st>>>(info_dev, n_frames, hist_in);
        h->acc_launches += 1;
    }
    CK(cudaStreamSynchronize(st));          // fg / mask are host vectors: the copies must be done before they go away
    CK(cudaGetLastError());
    x0_votes_end(h, ei);
    return SDV_OK;
}

int sdv_deint_pcm16x0(sdv_handle *h, const sdv_pcm16x0_config *cfg, const sdv_pcm16x0_subline *sublines_dev, int n_itl_blocks,
                      int16_t *samples_dev, uint8_t *sample_flags_dev, uint8_t *states_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!cfg||(n_itl_blocks<0)||(n_itl_blocks>(1<<25))) return fail(h, SDV_ERR_ARG, "sdv_deint_pcm16x0", cudaSuccess);
    if(n_itl_blocks==0) return SDV_OK;
    if(!sublines_dev||!samples_dev||((uintptr_t)sublines_dev%8)||((uintptr_t)samples_dev%4)||((uintptr_t)sample_flags_dev%2))
        return fail(h, SDV_ERR_ARG, "sdv_deint_pcm16x0: null or misaligned buffer", cudaSuccess);
    CK(cudaSetDevice(h->device));
    X0Cfg c; c.ignore_crc = cfg->ignore_crc; c.force_check = cfg->force_check; c.p_corr = cfg->p_corr;
    const int ei = cfg->ei_format ? 1 : 0;
    const long long nb = (long long)n_itl_blocks*(ei ? X0_BLOCKS_EI : X0_BLOCKS_ITL);
    pcm16x0_deint_kernel<<<(unsigned)((nb+255)/256), 256, 0, (cudaStream_t)cuda_stream>>>(sublines_dev, nb, c, ei, samples_dev, sample_flags_dev, states_dev);
    h->acc_launches += 1;
    CK(cudaGetLastError());
    return SDV_OK;
}

// Seam sweep launch: tasks_dev[n_tasks], every task up to max_n_pad paddings.
static int launch_seams(sdv_handle *h, const sdv_deint_config *cfg, int lim14, int lim16, const sdv_line_rec *recs_dev,
                        const SeamTask *tasks_dev, int n_tasks, int max_n_pad, sdv_stitch_stats *stats_dev, cudaStream_t st)
{
    SeamParams p;
    p.recs = recs_dev; p.tasks = tasks_dev; p.n_tasks = n_tasks;
    p.cfg = make_deint_cfg(cfg); p.cfg.force_check = 1;             // tryPadding forces the parity check
    p.lim14 = lim14; p.lim16 = lim16; p.out = stats_dev;
    for(int t0=0;t0<n_tasks;t0+=0x40000000)
    {
        const int nt = (n_tasks-t0<0x40000000) ? (n_tasks-t0) : 0x40000000;
        p.tasks = tasks_dev+t0;
        stc007_seam_kernel<<<dim3((unsigned)nt, (unsigned)max_n_pad), SEAM_THREADS, 0, st>>>(p);
        h->acc_launches += 1;
    }
    CK(cudaGetLastError());
    return SDV_OK;
}

int sdv_stc007_try_padding(sdv_handle *h, const sdv_deint_config *cfg, int max_unchecked_14bit, int max_unchecked_16bit,
                           const sdv_line_rec *recs_dev, const sdv_seam *seams_dev, int n_seams, int n_paddings,
                           sdv_stitch_stats *stats_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!cfg||(n_seams<0)||(n_paddings<1)||(n_paddings>64)||(cfg->res_mode>SDV_RES_MODE_16BIT)) return fail(h, SDV_ERR_ARG, "sdv_stc007_try_padding", cudaSuccess);
    if(n_seams==0) return SDV_OK;
    if(!recs_dev||!seams_dev||!stats_dev||((uintptr_t)recs_dev%16)) return fail(h, SDV_ERR_ARG, "sdv_stc007_try_padding: null or misaligned buffer", cudaSuccess);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    { int rc = ensure(h, (void **)&h->task_dev, &h->task_cap, (size_t)n_seams*sizeof(SeamTask)); if(rc) return rc; }
    seam_tasks_kernel<<<(unsigned)((n_seams+255)/256), 256, 0, st>>>(seams_dev, n_seams, n_paddings, h->task_dev);
    h->acc_launches += 1;
    return launch_seams(h, cfg, max_unchecked_14bit, max_unchecked_16bit, recs_dev, h->task_dev, n_seams, n_paddings, stats_dev, st);
}

// STC007DataStitcher::findPadding (stc007datastitcher.cpp:1743-2054): the sweep is one launch of the seam kernel for all
// seams x paddings; the decision over the (at most 32) statistics of a seam is host work (pad_decide, stc007_stitch_host.h).
int sdv_stc007_find_padding(sdv_handle *h, const sdv_deint_config *cfg, int video_std, int resolution_16bit,
                            int max_unchecked_14bit, int max_unchecked_16bit, const sdv_line_rec *recs_dev,
                            const sdv_seam *seams_host, int n_seams, sdv_padding *out_host, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!cfg||(n_seams<0)||(cfg->res_mode>SDV_RES_MODE_16BIT)||(video_std<0)||(video_std>2)) return fail(h, SDV_ERR_ARG, "sdv_stc007_find_padding", cudaSuccess);
    if(n_seams==0) return SDV_OK;
    if(!recs_dev||!seams_host||!out_host||((uintptr_t)recs_dev%16)) return fail(h, SDV_ERR_ARG, "sdv_stc007_find_padding: null or misaligned buffer", cudaSuccess);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const bool p_on = cfg->p_corr||cfg->q_corr, q_on = cfg->q_corr!=0;
    int max_padding = 32, lim = max_unchecked_14bit&0xFF;
    if(resolution_16bit||!q_on) { max_padding = 16; lim = max_unchecked_16bit&0xFF; }
    const int lpf = (video_std==1) ? ST_LINES_PF_PAL : ((video_std==2) ? ST_LINES_PF_NTSC : 0);
    std::vector<sdv_stitch_stats> stats;
    if(p_on)
    {
        const size_t seam_bytes = (size_t)n_seams*sizeof(sdv_seam), stat_bytes = (size_t)n_seams*max_padding*sizeof(sdv_stitch_stats);
        int rc = ensure(h, (void **)&h->pad_dev, &h->pad_cap, seam_bytes+stat_bytes+64);
        if(rc) return rc;
        sdv_seam *seams_dev = (sdv_seam *)h->pad_dev;
        sdv_stitch_stats *stats_dev = (sdv_stitch_stats *)(h->pad_dev+((seam_bytes+15)&~(size_t)15));
        CK(cudaMemcpyAsync(seams_dev, seams_host, seam_bytes, cudaMemcpyHostToDevice, st));
        if((rc = sdv_stc007_try_padding(h, cfg, max_unchecked_14bit, max_unchecked_16bit, recs_dev, seams_dev, n_seams, max_padding, stats_dev, st))) return rc;
        stats.resize((size_t)n_seams*max_padding);
        CK(cudaMemcpyAsync(stats.data(), stats_dev, stat_bytes, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    for(int s=0;s<n_seams;s++)
    {
        const PadDecision d = pad_decide(p_on ? &stats[(size_t)s*max_padding] : NULL, max_padding, seams_host[s].f1_size, lpf, lim, p_on);
        out_host[s].padding = d.padding; out_host[s].result = d.result; out_host[s].last_pad_counter = d.last_pad_counter;
    }
    return SDV_OK;
}

// ------------------------------------------------------------------------------------------------ STC-007 stitcher
namespace {
// Seam statistics for the host decision chain, computed by stc007_seam_kernel on demand and ahead of demand.
struct DevSeams : SeamOracle
{
    sdv_handle *h; const sdv_deint_config *cfg; int lim14, lim16; const sdv_line_rec *recs; int n_frames, H; cudaStream_t st;
    const FrameTrim *trims;                         // host copies, n_frames+1 (the last all zero: no frame behind the file)
    const u8 *step_res;                             // detected resolution: 4 modes per frame (ResChain::step), NULL = the preset of the call
    std::vector<int32_t> slot;                      // (frame*SEAM_KINDS+kind) -> sweep slot, -1 = not computed
    std::vector<sdv_stitch_stats> stats;            // 32 per slot
    std::unordered_map<uint64_t, uint8_t> tries;    // single paddings outside a sweep
    struct Req { int frame, kind, pad0, n_pad; };
    std::vector<Req> pending;
    int rc;

    SeamField field(int frame, int even) const
    {
        SeamField f; f.first = 0; f.size = 0; f.hole = ST_NO_HOLE;
        if(frame>=n_frames) return f;
        const FieldTrim &t = even ? trims[frame].even : trims[frame].odd;
        f.first = (u32)((size_t)frame*H+(even ? H/2 : 0)+t.first); f.size = t.data_lines; f.hole = t.hole;
        return f;
    }
    void seam_fields(int frame, int kind, SeamField *a, SeamField *b) const
    {
        static const int tab[SEAM_KINDS][3] = { {0, 0, 1}, {1, 0, 0}, {1, 1, 0}, {0, 1, 1}, {1, 1, 1}, {0, 1, 0} };   // field 1 parity, frame offset of field 2, field 2 parity
        *a = field(frame, tab[kind][0]); *b = field(frame+tab[kind][1], tab[kind][2]);
    }
    bool try_padding(int frame, int kind, int padding, uint8_t *result) override
    {
        const int32_t sl = slot[(size_t)frame*SEAM_KINDS+kind];
        if((sl>=0)&&(padding<32)) { *result = stats[(size_t)sl*32+padding].result; return true; }
        const uint64_t key = (((uint64_t)frame*SEAM_KINDS+kind)<<16)|(uint64_t)(padding&0xFFFF);
        auto it = tries.find(key);
        if(it!=tries.end()) { *result = it->second; return true; }
        Req r = { frame, kind, padding, 1 }; pending.push_back(r);
        return false;
    }
    bool sweep(int frame, int kind, const sdv_stitch_stats **stats32) override
    {
        const int32_t sl = slot[(size_t)frame*SEAM_KINDS+kind];
        if(sl>=0) { *stats32 = &stats[(size_t)sl*32]; return true; }
        Req r = { frame, kind, 0, 32 }; pending.push_back(r);
        return false;
    }
    // Run the requests on the device and file the answers.
    int compute(const std::vector<Req> &reqs)
    {
        if(reqs.empty()) return SDV_OK;
        std::vector<SeamTask> tasks(reqs.size());
        uint32_t n_out = 0; int max_pad = 1;
        for(size_t i=0;i<reqs.size();i++)
        {
            SeamTask t; seam_fields(reqs[i].frame, reqs[i].kind, &t.f1, &t.f2);
            t.pad0 = (u16)reqs[i].pad0; t.n_pad = (u16)reqs[i].n_pad; t.out = n_out; t.res1 = t.res2 = RES_ANY; t.pad_[0] = t.pad_[1] = 0;
            if(step_res)
            {   // the modes of the seam's two fields while frame [frame] is assembled
                static const int tab[SEAM_KINDS][3] = { {0, 0, 1}, {1, 0, 0}, {1, 1, 0}, {0, 1, 1}, {1, 1, 1}, {0, 1, 0} };
                const u8 *r = step_res+4*(size_t)reqs[i].frame; const int k = reqs[i].kind;
                t.res1 = r[tab[k][0]]; t.res2 = r[2*tab[k][1]+tab[k][2]];
            }
            n_out += (uint32_t)reqs[i].n_pad; if(reqs[i].n_pad>max_pad) max_pad = reqs[i].n_pad;
            tasks[i] = t;
        }
        int r;
        if((r = ensure(h, (void **)&h->task_dev, &h->task_cap, tasks.size()*sizeof(SeamTask)))) return r;
        if((r = ensure(h, (void **)&h->sstat_dev, &h->sstat_cap, (size_t)n_out*sizeof(sdv_stitch_stats)))) return r;
        if(cudaMemcpyAsync(h->task_dev, tasks.data(), tasks.size()*sizeof(SeamTask), cudaMemcpyHostToDevice, st)!=cudaSuccess) return SDV_ERR_CUDA;
        if((r = launch_seams(h, cfg, lim14, lim16, recs, h->task_dev, (int)tasks.size(), max_pad, h->sstat_dev, st))) return r;
        std::vector<sdv_stitch_stats> out(n_out);
        if(cudaMemcpyAsync(out.data(), h->sstat_dev, (size_t)n_out*sizeof(sdv_stitch_stats), cudaMemcpyDeviceToHost, st)!=cudaSuccess) return SDV_ERR_CUDA;
        if(cudaStreamSynchronize(st)!=cudaSuccess) return SDV_ERR_CUDA;
        for(size_t i=0;i<reqs.size();i++)
        {
            const Req &q = reqs[i];
            if((q.pad0==0)&&(q.n_pad==32))
            {
                const int32_t sl = (int32_t)(stats.size()/32);
                stats.insert(stats.end(), out.begin()+tasks[i].out, out.begin()+tasks[i].out+32);
                slot[(size_t)q.frame*SEAM_KINDS+q.kind] = sl;
            }
            else for(int k=0;k<q.n_pad;k++)
                tries[(((uint64_t)q.frame*SEAM_KINDS+q.kind)<<16)|(uint64_t)((q.pad0+k)&0xFFFF)] = out[tasks[i].out+k].result;
        }
        return SDV_OK;
    }
};

// The last [n] lines of the stream go into the handle for the next call (records + source frame / line number; a
// negative line number marks an empty line).
__global__ void save_carry_kernel(StitchMap m, long long first, int n, sdv_line_rec *recs_out, i32 *meta_out)
{
    const int i = blockIdx.x*blockDim.x+threadIdx.x;
    if(i>=n) return;
    int hint = (int)((first+i-m.n_carry-m.lead)/m.frame_len);
    const AsmLine l = stitch_line(m, first+i, &hint);
    sdv_line_rec r; memset(&r, 0, sizeof(r));
    if(l.rec) r = *l.rec;
    recs_out[i] = r;
    meta_out[2*i] = l.frame; meta_out[2*i+1] = l.rec ? l.line : (-l.line-1);
}
}   // namespace

int sdv_stc007_stitch_block_bound(int n_frames)
{
    if(n_frames<0) return SDV_ERR_ARG;
    const long long n = (long long)ST_LEAD_IN+ST_TAIL+(long long)n_frames*2*ST_LINES_PF_PAL;
    return (n>0x7FFFFFFF) ? SDV_ERR_ARG : (int)n;
}

int sdv_stc007_stitch_frames(sdv_handle *h, const sdv_deint_config *cfg, const sdv_stc007_stitch_config *scfg,
                             const sdv_line_rec *recs_dev, int n_frames, int H,
                             sdv_block_rec *blocks_dev, int16_t *samples_dev, uint8_t *sample_flags_dev,
                             int *n_blocks_out, int *n_frames_done, sdv_stc007_frame_info *info_host, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!cfg||!scfg||(n_frames<0)||(n_frames>(1<<22))||(H<2)||(H&1)||(H>2*SDV_MAX_H)||(scfg->video_std>2)||(scfg->field_order>2)||(cfg->res_mode>SDV_RES_MODE_16BIT)||(scfg->resolution_16bit>2))
        return fail(h, SDV_ERR_ARG, "sdv_stc007_stitch_frames", cudaSuccess);
    const bool res_auto = (scfg->resolution_16bit==2)&&!cfg->m2_format;     // (the reference does not detect the resolution of M2 tapes: 14 bit)
    const bool cwd = cfg->cwd!=0;
    std::vector<u8> cwd_patch;
    if((n_frames>0)&&(!recs_dev||((uintptr_t)recs_dev%16))) return fail(h, SDV_ERR_ARG, "sdv_stc007_stitch_frames: null or misaligned records", cudaSuccess);
    if((!scfg->file_start)&&(!h->carry_valid)) return fail(h, SDV_ERR_ARG, "sdv_stc007_stitch_frames: nothing to continue (file_start = 0 on a handle without an open file)", cudaSuccess);
    const int st_flags = (cwd ? SB_FLAG_CWD : 0)|(res_auto ? SB_FLAG_RES_AUTO : 0);
    if((!scfg->file_start)&&h->st_loaded&&(h->st_flags!=st_flags))
        return fail(h, SDV_ERR_ARG, "sdv_stc007_stitch_frames: the loaded state was saved with other CWD / resolution detection settings", cudaSuccess);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if(n_blocks_out) *n_blocks_out = 0;
    if(n_frames_done) *n_frames_done = 0;
    const int n_done = scfg->file_end ? n_frames : ((n_frames>0) ? (n_frames-1) : 0);
    int rc;
    // ---- trims of every frame (device), copied to the host for the decision chain
    std::vector<FrameTrim> trims((size_t)n_frames+1);
    std::vector<u8> field_res, step_res;
    memset(&trims[n_frames], 0, sizeof(FrameTrim)); trims[n_frames].odd.hole = trims[n_frames].even.hole = ST_NO_HOLE;
    if(n_frames>0)
    {
        if((rc = ensure(h, (void **)&h->trim_dev, &h->trim_cap, (size_t)n_frames*sizeof(FrameTrim)))) return rc;
        stc007_trim_kernel<<<n_frames, 128, 0, st>>>(recs_dev, n_frames, H, h->trim_dev);
        h->acc_launches += 1;
        CK(cudaMemcpyAsync(trims.data(), h->trim_dev, (size_t)n_frames*sizeof(FrameTrim), cudaMemcpyDeviceToHost, st));
        if(res_auto)
        {   // getFieldResolution of every field
            if((rc = ensure(h, (void **)&h->fres_dev, &h->fres_cap, 6*(size_t)n_frames+16))) return rc;
            stc007_fieldres_kernel<<<2*n_frames, 128, 0, st>>>(recs_dev, h->trim_dev, H, h->fres_dev);
            h->acc_launches += 1;
            field_res.resize(2*(size_t)n_frames);
            CK(cudaMemcpyAsync(field_res.data(), h->fres_dev, 2*(size_t)n_frames, cudaMemcpyDeviceToHost, st));
        }
        if(cwd)
        {   // frames with a line CWD may write into
            if((rc = ensure(h, (void **)&h->cwd_scan_dev, &h->cwd_scan_cap, (size_t)n_frames))) return rc;
            stc007_cwd_scan_kernel<<<n_frames, 128, 0, st>>>(recs_dev, H, h->cwd_scan_dev);
            h->acc_launches += 1;
            cwd_patch.resize((size_t)n_frames);
            CK(cudaMemcpyAsync(cwd_patch.data(), h->cwd_scan_dev, (size_t)n_frames, cudaMemcpyDeviceToHost, st));
        }
        CK(cudaStreamSynchronize(st));
        for(int f=0;f<n_frames;f++) if((trims[f].odd.holes>1)||(trims[f].even.holes>1))
            return fail(h, SDV_ERR_UNSUPPORTED, "sdv_stc007_stitch_frames: more than one service line inside the data lines of a field", cudaSuccess);
    }
    // ---- the decision chain
    Stitcher sx;
    sx.set.video_std = scfg->video_std; sx.set.field_order = scfg->field_order; sx.set.res16 = scfg->resolution_16bit ? 1 : 0;
    sx.set.p_corr = (cfg->p_corr||cfg->q_corr) ? 1 : 0; sx.set.q_corr = cfg->q_corr ? 1 : 0;
    sx.set.max_unch14 = scfg->max_unchecked_14bit; sx.set.max_unch16 = scfg->max_unchecked_16bit;
    sx.set.fix_cut_above = scfg->fix_cut_above; sx.set.mask_seams = scfg->mask_seams;
    if(scfg->file_start) { sx.st.reset(); h->st_frame_base = 0; h->st_countdown = 0; h->carry_valid = 0; h->st_res.reset(); h->cwd_carry_valid = 0; }
    else sx.st = h->st_carry;
    if(res_auto)
    {   // detectAudioResolution for every frame of the call: it needs nothing from the stitching decisions, and the seam sweeps need its modes
        ResChain rc2 = h->st_res;
        step_res.resize(4*(size_t)n_done+4);
        for(int f=0;f<n_done;f++)
        {
            const u8 bo = (f+1<n_frames) ? field_res[2*(size_t)f+2] : (u8)ST_RES_UNKNOWN, be = (f+1<n_frames) ? field_res[2*(size_t)f+3] : (u8)ST_RES_UNKNOWN;
            rc2.step(field_res[2*(size_t)f], field_res[2*(size_t)f+1], bo, be, &step_res[4*(size_t)f]);
        }
        if(!scfg->file_end) h->st_res = rc2;
    }
    DevSeams seams;
    seams.h = h; seams.cfg = cfg; seams.lim14 = scfg->max_unchecked_14bit; seams.lim16 = scfg->max_unchecked_16bit;
    seams.recs = recs_dev; seams.n_frames = n_frames; seams.H = H; seams.st = st; seams.trims = trims.data(); seams.rc = SDV_OK;
    seams.step_res = res_auto ? step_res.data() : NULL;
    seams.slot.assign((size_t)(n_frames+1)*SEAM_KINDS, -1);
    sx.seams = &seams;
    if((n_done>0)&&(sx.set.p_corr))
    {   // sweeps ahead of demand: the seams the chain asks for when nothing carries over from the frame before
        std::vector<DevSeams::Req> reqs;
        const bool preset = (scfg->field_order==ST_ORDER_TFF)||(scfg->field_order==ST_ORDER_BFF);
        for(int f=0;f<n_done;f++)
        {
            if(preset)
            {
                DevSeams::Req a = { f, Stitcher::inner_kind(scfg->field_order), 0, 32 }, b = { f, Stitcher::outer_kind(scfg->field_order, scfg->field_order), 0, 32 };
                reqs.push_back(a); reqs.push_back(b);
            }
            else for(int k=0;k<SEAM_KINDS;k++) { DevSeams::Req a = { f, k, 0, 32 }; reqs.push_back(a); }
        }
        if((rc = seams.compute(reqs))) return fail(h, rc, "sdv_stc007_stitch_frames: seam sweep", cudaGetLastError());
    }
    std::vector<FrameAsm> fa((size_t)n_done+1);
    std::vector<CwdStep> cwd_steps(cwd ? (size_t)n_done : 0);
    const int n_carry = scfg->file_start ? 0 : h->carry_valid;
    const int lead = scfg->file_start ? ST_LEAD_IN : 0;
    long long pos = lead;
    int frame_len = 2*ST_LINES_PF_NTSC, lead_line0 = 0;
    for(int f=0;f<n_done;f++)
    {
        int guard = 0;
        while(!sx.step(f, trims[f], trims[f+1], &fa[f], res_auto ? &step_res[4*(size_t)f] : NULL))
        {
            if((rc = seams.compute(seams.pending))) return fail(h, rc, "sdv_stc007_stitch_frames: seam sweep", cudaGetLastError());
            seams.pending.clear();
            if(++guard>64) return fail(h, SDV_ERR_CUDA, "sdv_stc007_stitch_frames: decision chain does not settle", cudaSuccess);
        }
        seams.pending.clear();
        fa[f].start = (i32)pos; pos += fa[f].total;
        const FrameSt &r = sx.st.f0;
        if(cwd)
        {
            CwdStep cs; cs.begin = (i32)(n_carry+fa[f].start); cs.end = cs.begin+fa[f].total+(((f==n_done-1)&&scfg->file_end) ? ST_TAIL : 0);
            cwd_next_field(r, trims[f+1], (size_t)(f+1)*H, H, &cs);
            cwd_steps[f] = cs;
        }
        if(f==0)
        {
            const int T = (r.video_std==ST_VID_PAL) ? ST_LINES_PF_PAL : ST_LINES_PF_NTSC;
            frame_len = 2*T; lead_line0 = 2*T-2*ST_LEAD_IN;
        }
        if(info_host)
        {
            sdv_stc007_frame_info o; memset(&o, 0, sizeof(o));
            o.start = fa[f].start+n_carry; o.pre = fa[f].pre; o.n1 = fa[f].n1; o.inner = fa[f].inner; o.n2 = fa[f].n2; o.outer = fa[f].outer;
            o.skip1 = fa[f].skip1; o.skip2 = fa[f].skip2;
            o.odd_top = trims[f].odd.top; o.odd_bottom = trims[f].odd.bottom; o.even_top = trims[f].even.top; o.even_bottom = trims[f].even.bottom;
            o.odd_data_lines = trims[f].odd.data_lines; o.even_data_lines = trims[f].even.data_lines;
            o.odd_valid_lines = trims[f].odd.valid_lines; o.even_valid_lines = trims[f].even.valid_lines;
            o.inner_padding = r.inner_pad; o.outer_padding = r.outer_pad; o.field_order = r.order; o.video_std = r.video_std;
            o.flags = (uint8_t)((r.inner_ok ? SDV_FA_INNER_OK : 0)|(r.outer_ok ? SDV_FA_OUTER_OK : 0)|(r.inner_silence ? SDV_FA_INNER_SILENCE : 0)
                      |(r.outer_silence ? SDV_FA_OUTER_SILENCE : 0)|(r.order_guessed ? SDV_FA_ORDER_GUESSED : 0)
                      |((fa[f].mask&1) ? SDV_FA_MASK_INNER : 0)|((fa[f].mask&2) ? SDV_FA_MASK_PREV_OUTER : 0));
            o.odd_res_mode = res_auto ? r.odd_res : cfg->res_mode; o.even_res_mode = res_auto ? r.even_res : cfg->res_mode;
            info_host[f] = o;
        }
    }
    // ---- the stream and its blocks
    const int tail = scfg->file_end ? ST_TAIL : 0;
    const long long n_lines = (long long)n_carry+pos+tail;
    const long long n_blocks = (n_lines>ST_TAIL) ? (n_lines-ST_TAIL) : 0;
    if(n_blocks>0x7FFFFFFF) return fail(h, SDV_ERR_ARG, "sdv_stc007_stitch_frames: too many blocks for one call", cudaSuccess);
    if((n_blocks>0)&&((!samples_dev&&!sample_flags_dev&&!blocks_dev)||((uintptr_t)samples_dev%4)||((uintptr_t)sample_flags_dev%2)))
        return fail(h, SDV_ERR_ARG, "sdv_stc007_stitch_frames: null or misaligned output", cudaSuccess);
    if((rc = ensure(h, (void **)&h->fa_dev, &h->fa_cap, ((size_t)n_done+1)*sizeof(FrameAsm)))) return rc;
    if(n_done>0) CK(cudaMemcpyAsync(h->fa_dev, fa.data(), (size_t)n_done*sizeof(FrameAsm), cudaMemcpyHostToDevice, st));
    bool cwd_last_dirty = false;
    StitchMap m; memset(&m, 0, sizeof(m));
    m.recs = recs_dev; m.fa = h->fa_dev; m.n_frames = n_done; m.H = H;
    m.lead = lead; m.lead_line0 = lead_line0; m.tail = tail;
    m.carry = h->carry_dev[h->carry_cur]; m.carry_meta = h->carry_meta_dev[h->carry_cur]; m.n_carry = n_carry;
    m.frame_base = h->st_frame_base; m.frame_len = frame_len; m.n_lines = n_lines;
    if(res_auto&&(n_done>0))
    {
        CK(cudaMemcpyAsync(h->fres_dev+2*(size_t)n_frames, step_res.data(), 4*(size_t)n_done, cudaMemcpyHostToDevice, st));
        m.step_res = h->fres_dev+2*(size_t)n_frames;
        if(scfg->file_start) m.f0_res[0] = m.f0_res[1] = step_res[fa[0].first_even ? 1 : 0];      // fillFrameForOutput at a file start (stc007datastitcher.cpp:4716-4723)
        else { m.f0_res[0] = h->st_carry.f0.odd_res; m.f0_res[1] = h->st_carry.f0.even_res; }
    }
    if(n_blocks>0)
    {
        DeintScratch sc;
        if((rc = deint_scratch(h, n_blocks, cfg->broken_mask_dur, &sc))) return rc;
        StitchDeintParams p;
        p.map = m; p.n_blocks = n_blocks; p.cfg = make_deint_cfg(cfg);
        if(cwd&&!blocks_dev)
        {   // CWD: the countdown windows are applied to stored blocks (the lines behind them were patched), so the records are kept
            if((rc = ensure(h, (void **)&h->blk_scratch, &h->blk_scratch_cap, (size_t)n_blocks*sizeof(sdv_block_rec)))) return rc;
            blocks_dev = h->blk_scratch;
        }
        p.blocks = blocks_dev; p.samples = samples_dev; p.sflags = sample_flags_dev;
        p.broken_bits = sc.bits; p.broken_sum = sc.sum;
        CK(cudaMemsetAsync(sc.sum, 0, (size_t)((n_blocks+1023)>>10), st));
        timing_flush(h, 1);
        cudaEventRecord(h->ev[2], st);
        stc007_stitch_deint_kernel<<<(unsigned)((n_blocks+255)/256), 256, 0, st>>>(p);
        cudaEventRecord(h->ev[3], st);
        h->ev_set[1] = 1; h->ev_units[1] = (uint64_t)n_blocks; h->acc_launches += 1;
        cwd_last_dirty = false;
        if(cwd&&(n_done>0))
        {   // the frames CWD can touch, chain by chain: their blocks are computed again from the patched queue
            std::vector<int> chains; std::vector<u8> dirty;
            cwd_plan_chains(cwd_patch.data(), fa.data(), n_done, (!scfg->file_start)&&h->cwd_carry_valid, &chains, &dirty);
            cwd_last_dirty = dirty[(size_t)n_done-1]!=0;
            if(!chains.empty())
            {
                int longest = 0, n_dirty = 0;
                for(size_t k=0;k<chains.size();k+=2) { if(chains[k+1]>longest) longest = chains[k+1]; n_dirty += chains[k+1]; }
                static const int spec_env = getenv("SDV_CWD_SPECULATE") ? atoi(getenv("SDV_CWD_SPECULATE")) : -1;      // tuning knob: 0 never, 1 always
                const bool speculate = (spec_env>=0) ? (spec_env!=0) : (longest>=8);
                const size_t step_bytes = (size_t)n_done*sizeof(CwdStep);
                // plan area: steps | chains or frame list | per-step mode | verify list | verify result
                const size_t list_cap = (size_t)(speculate ? 2*n_dirty : (int)chains.size())*sizeof(int);
                const size_t need = step_bytes+list_cap+(size_t)n_done+(size_t)n_dirty*sizeof(int)+(size_t)n_dirty+64;
                if((rc = ensure(h, (void **)&h->cwd_plan_dev, &h->cwd_plan_cap, need))) return rc;
                u8 *plan = h->cwd_plan_dev;
                int *list_dev = (int *)(plan+step_bytes);
                u8 *mode_dev = plan+step_bytes+list_cap;
                int *vlist_dev = (int *)(plan+((step_bytes+list_cap+(size_t)n_done+15)&~(size_t)15));
                u8 *vok_dev = (u8 *)(vlist_dev+n_dirty);
                CK(cudaMemcpyAsync(plan, cwd_steps.data(), step_bytes, cudaMemcpyHostToDevice, st));
                CK(cudaMemsetAsync(h->cwd_status, 0, sizeof(int), st));
                CwdParams cp; memset(&cp, 0, sizeof(cp));
                cp.map = m; cp.steps = (const CwdStep *)plan; cp.chains = list_dev;
                cp.cfg = p.cfg; cp.n_blocks = n_blocks;
                cp.blocks = blocks_dev; cp.samples = samples_dev; cp.sflags = sample_flags_dev;
                cp.broken_bits = (cfg->broken_mask_dur>0) ? sc.bits : NULL; cp.broken_sum = sc.sum;
                cp.carry_in = ((!scfg->file_start)&&h->cwd_carry_valid) ? h->cwd_carry[h->carry_cur] : NULL;
                cp.carry_out = h->cwd_carry[h->carry_cur^1]; cp.carry_out_step = ((!scfg->file_end)&&cwd_last_dirty) ? (n_done-1) : -1;
                cp.status = h->cwd_status;
                if(!speculate)
                {
                    CK(cudaMemcpyAsync(list_dev, chains.data(), chains.size()*sizeof(int), cudaMemcpyHostToDevice, st));
                    stc007_cwd_chain_kernel<<<(unsigned)(chains.size()/2), CWD_THREADS, 0, st>>>(cp);
                    h->acc_launches += 1;
                }
                else
                {   // every dirty frame at once from the lines as they are on the tape, then again those whose predecessor left other
                    // lines than they took (see CwdParams); a frame that is first in its chain takes exact input by construction
                    if((rc = ensure(h, (void **)&h->cwd_spec_dev, &h->cwd_spec_cap, (size_t)n_done*(2*112*sizeof(CwdLine)+2*sizeof(u16))+64))) return rc;
                    cp.step_out = (CwdLine *)h->cwd_spec_dev; cp.step_used = cp.step_out+(size_t)n_done*112;
                    cp.step_n = (u16 *)(cp.step_used+(size_t)n_done*112); cp.step_mode = mode_dev; cp.step_first = NULL;
                    std::vector<int> frames, vlist; std::vector<u8> mode((size_t)n_done, 0), vok;
                    for(size_t k=0;k<chains.size();k+=2) for(int q=0;q<chains[k+1];q++)
                    {
                        frames.push_back(chains[k]+q); frames.push_back(1);
                        if(q>0) vlist.push_back(chains[k]+q);
                    }
                    CK(cudaMemcpyAsync(vlist_dev, vlist.data(), vlist.size()*sizeof(int), cudaMemcpyHostToDevice, st));
                    vok.resize(vlist.size());
                    int rounds = 0;
                    for(;;)
                    {
                        CK(cudaMemcpyAsync(list_dev, frames.data(), frames.size()*sizeof(int), cudaMemcpyHostToDevice, st));
                        CK(cudaMemcpyAsync(mode_dev, mode.data(), (size_t)n_done, cudaMemcpyHostToDevice, st));
                        stc007_cwd_chain_kernel<<<(unsigned)(frames.size()/2), CWD_THREADS, 0, st>>>(cp);
                        h->acc_launches += 1;
                        if(vlist.empty()) break;
                        cwd_verify_kernel<<<(unsigned)vlist.size(), 128, 0, st>>>(vlist_dev, (int)vlist.size(), cp.step_out, cp.step_used, cp.step_n, vok_dev);
                        h->acc_launches += 1;
                        CK(cudaMemcpyAsync(vok.data(), vok_dev, vok.size(), cudaMemcpyDeviceToHost, st));
                        CK(cudaStreamSynchronize(st));
                        frames.clear();
                        for(size_t k=0;k<vlist.size();k++) if(!vok[k]) { frames.push_back(vlist[k]); frames.push_back(1); mode[(size_t)vlist[k]] = 1; }
                        if(frames.empty()) break;
                        if(++rounds>n_dirty+2) return fail(h, SDV_ERR_CUDA, "sdv_stc007_stitch_frames: CWD walk does not settle", cudaSuccess);
                    }
                    h->stats.frames_skipped = (uint64_t)rounds;
                }
                h->stats.reserved = (uint32_t)(chains.size()/2);
            }
        }
        if(cfg->broken_mask_dur>0)
        {
            WindowParams wp; memset(&wp, 0, sizeof(wp));
            wp.from_records = cwd ? 1 : 0;
            wp.stitched = 1; wp.smap = m; wp.n_blocks = n_blocks; wp.cfg = p.cfg;
            wp.blocks = blocks_dev; wp.samples = samples_dev; wp.sflags = sample_flags_dev;
            if((rc = run_windows(h, sc, wp, cfg->broken_mask_dur, scfg->file_start ? 0 : h->st_countdown, st))) return rc;
        }
    }
    // ---- what the next call continues from
    if(!scfg->file_end)
    {
        const int keep = (int)((n_lines<ST_TAIL) ? n_lines : ST_TAIL);
        const int nxt = h->carry_cur^1;
        if(keep>0) save_carry_kernel<<<1, 128, 0, st>>>(m, n_lines-keep, keep, h->carry_dev[nxt], h->carry_meta_dev[nxt]);
        h->acc_launches += 1;
        CK(cudaMemcpyAsync(h->win_state_host, h->win_state, 4*sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        h->carry_cur = nxt; h->carry_valid = keep;
        h->cwd_carry_valid = (cwd&&cwd_last_dirty&&(n_blocks>0)) ? 1 : ((n_done>0) ? 0 : h->cwd_carry_valid);
        h->st_carry = sx.st; h->st_frame_base += n_done;
        h->st_countdown = ((n_blocks>0)&&(cfg->broken_mask_dur>0)) ? h->win_state_host[1] : h->st_countdown;
        h->st_flags = st_flags;
    }
    else
    {
        CK(cudaStreamSynchronize(st));
        h->carry_valid = 0; h->st_countdown = 0; h->cwd_carry_valid = 0;
    }
    h->st_loaded = 0;
    CK(cudaGetLastError());
    if(cwd)
    {
        int stt = 0;
        CK(cudaMemcpy(&stt, h->cwd_status, sizeof(int), cudaMemcpyDeviceToHost));
        if(stt) return fail(h, SDV_ERR_UNSUPPORTED, "sdv_stc007_stitch_frames: a frame too long for the CWD queue", cudaSuccess);
    }
    if(n_blocks_out) *n_blocks_out = (int)n_blocks;
    if(n_frames_done) *n_frames_done = n_done;
    return SDV_OK;
}

// ---- the open file of the stitcher as a blob (layout: SB_* in stc007_stitch.cuh)
static_assert((sizeof(CwdLine)==32)&&(offsetof(CwdLine, frame)==28)&&(sizeof(sdv_line_rec)==32), "blob layout of the carried lines");
static void sb_put(StitchBlobHdr *o, int at, const void *p, size_t n) { memcpy((u8 *)o->w+at, p, n); }
static const u8 *sb_at(const StitchBlobHdr &o, int at) { return (const u8 *)o.w+at; }

static StitchBlobHdr stitch_state_encode(const sdv_handle *h)
{
    StitchBlobHdr o; memset(&o, 0, sizeof(o));
    const u32 magic = SB_MAGIC, size = SB_BYTES; const u16 version = SB_VERSION, flags = (u16)h->st_flags;
    const i32 n_carry = h->carry_valid, n_cwd = h->cwd_carry_valid ? h->carry_valid : 0, countdown = h->st_countdown;
    sb_put(&o, SBH_MAGIC, &magic, 4); sb_put(&o, SBH_VERSION, &version, 2); sb_put(&o, SBH_FLAGS, &flags, 2); sb_put(&o, SBH_SIZE, &size, 4);
    sb_put(&o, SBH_CARRY, &n_carry, 4); sb_put(&o, SBH_CWD_VALID, &n_cwd, 4); sb_put(&o, SBH_COUNTDOWN, &countdown, 4);
    const FrameSt &f = h->st_carry.f0;
    const u16 w16[4] = { f.odd_lines, f.even_lines, f.inner_pad, f.outer_pad };
    const u8 w8[13] = { f.order, (u8)f.order_preset, (u8)f.order_guessed, f.video_std, (u8)f.std_preset, (u8)f.inner_ok, (u8)f.outer_ok,
                        (u8)f.inner_silence, (u8)f.outer_silence, f.tff_cnt, f.bff_cnt, f.odd_res, f.even_res };
    sb_put(&o, SBH_F0, w16, 8); sb_put(&o, SBH_F0+8, w8, 13);
    sb_put(&o, SBH_LAST_PAD, &h->st_carry.last_pad_counter, 1);
    u8 *order = (u8 *)o.w+SBH_ORDER, *res = (u8 *)o.w+SBH_RES;     // the rings from their oldest entry on, position 0
    for(int i=0;i<65;i++) { order[i] = h->st_carry.order_hist[(h->st_carry.order_pos+i)%65]; res[i] = h->st_res.hist[(h->st_res.pos+i)%65]; }
    return o;
}

// Header -> handle state; false for a blob this build did not write (nothing is changed then).
static bool stitch_state_decode(const StitchBlobHdr &o, sdv_handle *h)
{
    u32 magic, size; u16 version, flags; i32 n_carry, n_cwd, countdown;
    memcpy(&magic, sb_at(o, SBH_MAGIC), 4); memcpy(&version, sb_at(o, SBH_VERSION), 2); memcpy(&flags, sb_at(o, SBH_FLAGS), 2);
    memcpy(&size, sb_at(o, SBH_SIZE), 4); memcpy(&n_carry, sb_at(o, SBH_CARRY), 4); memcpy(&n_cwd, sb_at(o, SBH_CWD_VALID), 4);
    memcpy(&countdown, sb_at(o, SBH_COUNTDOWN), 4);
    if((magic!=SB_MAGIC)||(version!=SB_VERSION)||(size!=SB_BYTES)||(flags>3)) return false;
    if((n_carry<1)||(n_carry>ST_TAIL)||((n_cwd!=0)&&(n_cwd!=n_carry))||((n_cwd!=0)&&!(flags&SB_FLAG_CWD))||(countdown<0)||(countdown>255)) return false;
    u16 w16[4]; u8 w8[13];
    memcpy(w16, sb_at(o, SBH_F0), 8); memcpy(w8, sb_at(o, SBH_F0+8), 13);
    if((w8[0]>2)||(w8[3]>2)||(w8[11]>SDV_RES_MODE_16BIT)||(w8[12]>SDV_RES_MODE_16BIT)) return false;
    for(int i : {1, 2, 4, 5, 6, 7, 8}) if(w8[i]>1) return false;
    const u8 *order = sb_at(o, SBH_ORDER), *res = sb_at(o, SBH_RES);
    for(int i=0;i<65;i++) if((order[i]>2)||(res[i]>2)) return false;
    FrameSt &f = h->st_carry.f0;
    f.odd_lines = w16[0]; f.even_lines = w16[1]; f.inner_pad = w16[2]; f.outer_pad = w16[3];
    f.order = w8[0]; f.order_preset = w8[1]; f.order_guessed = w8[2]; f.video_std = w8[3]; f.std_preset = w8[4]; f.inner_ok = w8[5];
    f.outer_ok = w8[6]; f.inner_silence = w8[7]; f.outer_silence = w8[8]; f.tff_cnt = w8[9]; f.bff_cnt = w8[10]; f.odd_res = w8[11]; f.even_res = w8[12];
    h->st_carry.last_pad_counter = *sb_at(o, SBH_LAST_PAD);
    memcpy(h->st_carry.order_hist, order, 65); h->st_carry.order_pos = 0;
    memcpy(h->st_res.hist, res, 65); h->st_res.pos = 0;
    h->st_countdown = countdown; h->carry_valid = n_carry; h->cwd_carry_valid = n_cwd ? 1 : 0;
    h->st_frame_base = 0; h->st_flags = flags; h->st_loaded = 1;
    return true;
}

int sdv_stc007_stitch_state_bytes(void) { return SB_BYTES; }

int sdv_stc007_stitch_state_save(sdv_handle *h, void *state_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!state_dev||((uintptr_t)state_dev%4)) return fail(h, SDV_ERR_ARG, "sdv_stc007_stitch_state_save: null or misaligned state buffer", cudaSuccess);
    if(!h->carry_valid) return fail(h, SDV_ERR_ARG, "sdv_stc007_stitch_state_save: no open file on the handle", cudaSuccess);
    CK(cudaSetDevice(h->device));
    const StitchBlobHdr hdr = stitch_state_encode(h);
    const int c = h->carry_cur;
    stitch_state_pack_kernel<<<(SB_BYTES/4+255)/256, 256, 0, (cudaStream_t)cuda_stream>>>(hdr, (const u32 *)h->carry_dev[c], h->carry_meta_dev[c],
        (const u32 *)h->cwd_carry[c], h->carry_valid, h->cwd_carry_valid ? h->carry_valid : 0, h->st_frame_base+1, (u32 *)state_dev);
    h->acc_launches += 1;
    CK(cudaGetLastError());
    return SDV_OK;
}

int sdv_stc007_stitch_state_load(sdv_handle *h, const void *state_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!state_dev||((uintptr_t)state_dev%4)) return fail(h, SDV_ERR_ARG, "sdv_stc007_stitch_state_load: null or misaligned state buffer", cudaSuccess);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    StitchBlobHdr hdr;
    CK(cudaMemcpyAsync(&hdr, state_dev, sizeof(hdr), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if(!stitch_state_decode(hdr, h)) return fail(h, SDV_ERR_ARG, "sdv_stc007_stitch_state_load: not a stitcher state of this version", cudaSuccess);
    const int c = h->carry_cur;
    stitch_state_unpack_kernel<<<(SB_BYTES/4+255)/256, 256, 0, st>>>((const u32 *)state_dev, (u32 *)h->carry_dev[c], h->carry_meta_dev[c], (u32 *)h->cwd_carry[c], 1);
    h->acc_launches += 1;
    CK(cudaStreamSynchronize(st));
    return SDV_OK;
}

int sdv_stc007_block_count(const sdv_stc007_geometry *geo, int n_frames)
{
    if(!geo||(n_frames<0)) return SDV_ERR_ARG;
    long long n = (long long)geo->lead_in+(long long)n_frames*2*geo->lines_per_field;
    return (n>0x7FFFFFFF) ? SDV_ERR_ARG : (int)n;
}

int sdv_stc007_frames_to_samples(sdv_handle *h, const sdv_deint_config *cfg, const sdv_stc007_geometry *geo,
                                 const sdv_line_rec *recs_dev, int n_frames, int H,
                                 sdv_block_rec *blocks_dev, int16_t *samples_dev, uint8_t *sample_flags_dev, void *cuda_stream)
{
    return sdv_stc007_shard_to_samples(h, cfg, geo, recs_dev, n_frames, H, NULL, blocks_dev, samples_dev, sample_flags_dev, cuda_stream);
}

int sdv_stc007_shard_to_samples(sdv_handle *h, const sdv_deint_config *cfg, const sdv_stc007_geometry *geo,
                                const sdv_line_rec *recs_dev, int n_frames, int H, const sdv_line_rec *halo_dev,
                                sdv_block_rec *blocks_dev, int16_t *samples_dev, uint8_t *sample_flags_dev, void *cuda_stream)
{
    if(!h) return SDV_ERR_ARG;
    if(!cfg||!geo||(!recs_dev&&(n_frames>0))||((uintptr_t)recs_dev%16)||(n_frames<0)||(H<2)||(H&1)||(geo->lines_per_field<H/2)||(cfg->res_mode>SDV_RES_MODE_16BIT))
        return fail(h, SDV_ERR_ARG, "sdv_stc007_frames_to_samples", cudaSuccess);
    CK(cudaSetDevice(h->device));
    const long long nb = (long long)geo->lead_in+(long long)n_frames*2*geo->lines_per_field;
    AsmMap m; memset(&m, 0, sizeof(m));
    m.recs = recs_dev; m.geo = 1; m.lead_in = geo->lead_in; m.lpf = geo->lines_per_field; m.hf = H/2; m.H = H;
    m.n_fields = (long long)n_frames*2; m.n_lines = nb+112; m.halo = halo_dev;
    if((uintptr_t)halo_dev%16) return fail(h, SDV_ERR_ARG, "sdv_stc007_shard_to_samples: misaligned halo", cudaSuccess);
    return run_deint(h, cfg, m, nb, blocks_dev, samples_dev, sample_flags_dev, (cudaStream_t)cuda_stream);
}

int sdv_stc007_decode_tape_host(sdv_handle *h, const sdv_bin_config *bcfg, const sdv_deint_config *dcfg,
                                const sdv_stc007_geometry *geo, const uint8_t *luma_host, int n_frames, int H, int W,
                                int16_t *samples_host, uint8_t *flags_host, sdv_line_rec *recs_host)
{
    if(!h) return SDV_ERR_ARG;
    if(!bcfg||!dcfg||!geo||!luma_host||!samples_host||(n_frames<0)) return fail(h, SDV_ERR_ARG, "sdv_stc007_decode_tape_host", cudaSuccess);
    CK(cudaSetDevice(h->device));
    const size_t luma_bytes = (size_t)n_frames*H*W;
    const long long nb = (long long)geo->lead_in+(long long)n_frames*2*geo->lines_per_field;
    int rc;
    if((rc = ensure(h, (void **)&h->luma_dev, &h->luma_cap, luma_bytes+64))) return rc;
    if((rc = ensure(h, (void **)&h->recs_dev, &h->recs_cap, (size_t)n_frames*H*sizeof(sdv_line_rec)+64))) return rc;
    if(h->smp_cap<(size_t)nb)
    {
        cudaFree(h->smp_dev); cudaFree(h->sfl_dev); h->smp_dev = NULL; h->sfl_dev = NULL; h->smp_cap = 0;
        CK(cudaMalloc(&h->smp_dev, (size_t)nb*6*sizeof(i16)+64));
        CK(cudaMalloc(&h->sfl_dev, (size_t)nb*6+64));
        h->smp_cap = (size_t)nb;
    }
    cudaStream_t st = h->stream;
    CK(cudaMemcpyAsync(h->luma_dev, luma_host, luma_bytes, cudaMemcpyHostToDevice, st));
    if((rc = sdv_bin_decode_frames(h, bcfg, h->luma_dev, n_frames, H, W, W, h->recs_dev, NULL, st))) return rc;
    if((rc = sdv_stc007_frames_to_samples(h, dcfg, geo, h->recs_dev, n_frames, H, NULL, h->smp_dev, flags_host ? h->sfl_dev : NULL, st))) return rc;
    CK(cudaMemcpyAsync(samples_host, h->smp_dev, (size_t)nb*6*sizeof(i16), cudaMemcpyDeviceToHost, st));
    if(flags_host) CK(cudaMemcpyAsync(flags_host, h->sfl_dev, (size_t)nb*6, cudaMemcpyDeviceToHost, st));
    if(recs_host) CK(cudaMemcpyAsync(recs_host, h->recs_dev, (size_t)n_frames*H*sizeof(sdv_line_rec), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SDV_OK;
}

// Host-buffer entry points for PCM-1 and PCM-16x0 (SI): H2D luma, line decode, frame assembly + deinterleave, D2H samples.
static int decode_tape_host_fmt(sdv_handle *h, int x0, const sdv_bin_config *bcfg, const sdv_pcm1_stitch_config *p1cfg,
                                const sdv_pcm16x0_config *xcfg, const sdv_pcm16x0_geometry *xgeo, const uint8_t *luma_host, int n_frames,
                                int H, int W, int16_t *samples_host, uint8_t *flags_host, sdv_line_rec *recs_host)
{
    CK(cudaSetDevice(h->device));
    const size_t luma_bytes = (size_t)n_frames*H*W;
    const size_t n_recs = (size_t)n_frames*H*(x0 ? 3 : 1);
    const size_t n_smp = (size_t)n_frames*2*1470;               // 735 sample pairs per field in both formats
    int rc;
    if((rc = ensure(h, (void **)&h->luma_dev, &h->luma_cap, luma_bytes+64))) return rc;
    if((rc = ensure(h, (void **)&h->recs_dev, &h->recs_cap, n_recs*sizeof(sdv_line_rec)+64))) return rc;
    if(h->smp_cap<(n_smp+5)/6)
    {
        cudaFree(h->smp_dev); cudaFree(h->sfl_dev); h->smp_dev = NULL; h->sfl_dev = NULL; h->smp_cap = 0;
        CK(cudaMalloc(&h->smp_dev, n_smp*sizeof(i16)+64));
        CK(cudaMalloc(&h->sfl_dev, n_smp+64));
        h->smp_cap = (n_smp+5)/6;
    }
    cudaStream_t st = h->stream;
    CK(cudaMemcpyAsync(h->luma_dev, luma_host, luma_bytes, cudaMemcpyHostToDevice, st));
    if((rc = sdv_bin_decode_frames(h, bcfg, h->luma_dev, n_frames, H, W, W, h->recs_dev, NULL, st))) return rc;
    if(x0) rc = sdv_pcm16x0_frames_to_samples(h, xcfg, xgeo, h->recs_dev, n_frames, H, NULL, h->smp_dev, flags_host ? h->sfl_dev : NULL, st);
    else rc = sdv_pcm1_frames_to_samples(h, p1cfg, h->recs_dev, n_frames, H, h->smp_dev, flags_host ? h->sfl_dev : NULL, NULL, st);
    if(rc) return rc;
    CK(cudaMemcpyAsync(samples_host, h->smp_dev, n_smp*sizeof(i16), cudaMemcpyDeviceToHost, st));
    if(flags_host) CK(cudaMemcpyAsync(flags_host, h->sfl_dev, n_smp, cudaMemcpyDeviceToHost, st));
    if(recs_host) CK(cudaMemcpyAsync(recs_host, h->recs_dev, n_recs*sizeof(sdv_line_rec), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SDV_OK;
}

int sdv_pcm1_decode_tape_host(sdv_handle *h, const sdv_bin_config *bcfg, const sdv_pcm1_stitch_config *scfg, const uint8_t *luma_host,
                              int n_frames, int H, int W, int16_t *samples_host, uint8_t *flags_host, sdv_line_rec *recs_host)
{
    if(!h) return SDV_ERR_ARG;
    if(!bcfg||!scfg||!luma_host||!samples_host||(n_frames<0)||(bcfg->pcm_type!=SDV_TYPE_PCM1)) return fail(h, SDV_ERR_ARG, "sdv_pcm1_decode_tape_host", cudaSuccess);
    if(n_frames==0) return SDV_OK;
    return decode_tape_host_fmt(h, 0, bcfg, scfg, NULL, NULL, luma_host, n_frames, H, W, samples_host, flags_host, recs_host);
}

int sdv_pcm16x0_decode_tape_host(sdv_handle *h, const sdv_bin_config *bcfg, const sdv_pcm16x0_config *dcfg, const sdv_pcm16x0_geometry *geo,
                                 const uint8_t *luma_host, int n_frames, int H, int W, int16_t *samples_host, uint8_t *flags_host,
                                 sdv_line_rec *recs_host)
{
    if(!h) return SDV_ERR_ARG;
    if(!bcfg||!dcfg||!geo||!luma_host||!samples_host||(n_frames<0)||(bcfg->pcm_type!=SDV_TYPE_PCM16X0)) return fail(h, SDV_ERR_ARG, "sdv_pcm16x0_decode_tape_host", cudaSuccess);
    if(n_frames==0) return SDV_OK;
    return decode_tape_host_fmt(h, 1, bcfg, NULL, dcfg, geo, luma_host, n_frames, H, W, samples_host, flags_host, recs_host);
}

}   // extern "C"
