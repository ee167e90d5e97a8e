// stc007_bulk.cuh -- the HBM-bound pass of the STC-007 line decode (device only).
//
// What it computes: for every video line of the given frames, the preset-only decode the reference takes on a good
// tape (Binarizer::processLine STG_INPUT_ALL -> readPCMdata first candidate -> STG_DATA_OK, binarizer.cpp:774-931,
// 7695-8055) with the chain's steady-state reference level and data coordinates, plus the per-field rules
// VideoToDigital applies to a valid line (first PCM line of a field, duplicate line; videotodigital.cpp:1159-1278).
// A field in which every line decodes this way is flagged clean; everything else is redone by stc007_chain_kernel.
//
// How: one LANE per video line, 32 consecutive rows of a frame per warp step, staged in shared memory by the per-warp
// ring of bulk_ring.cuh (one 1-D bulk copy per step).  Each lane walks the 128 bit-cell centres of its row: one byte load per cell (the cell positions are
// launch constants read from the kernel parameter bank), and two funnel-shift registers accumulate "pixel > ref" and
// "pixel >= ref" MSB-first, which is already the bit order of the PCM words.  Cells sitting exactly on the reference
// level keep the previous bit (the reference's level hysteresis at depth 0): resolved per lane as a 128-bit carry
// chain.  CRCC by a 256-entry table in shared memory, 14 steps.  Two 16-byte stores per lane write the line record.
#pragma once
#include "bulk_ring.cuh"
#include "stc007_chain.cuh"
#include "stc007_deint.cuh"

namespace sdv {

__constant__ u16 c_crc8[3*256];     // [0..255]: CRC-16 CCITT byte table (CRC, init 0, of the byte x);
                                    // [256..511] / [512..767]: the CRC state x / x<<8 advanced over 7 zero bytes
enum { BULK_SMEM_HEADER = BULK_BAR_BYTES+3*512 };

struct BulkParams
{
    const u8 *luma; int H, W; size_t stride;
    int f0, n_frames;               // frames [f0, f0+n_frames)
    u8 ref, black, white, line_dup; Coord coords;   // line_dup: bit 0 = duplicate-line check, bit 1 = M2 tape
    sdv_line_rec *recs; sdv_line_aux *aux;
    u8 *clean;                      // [2*total frames] per field: 1 = every line of the field was taken by this kernel
    int *first_unclean;             // atomicMin of the frames with a field that is not clean
    int use_tma, warps; u32 slot_bytes;
    u32 pos[BITS_PCM_DATA];         // pixel of each bit cell centre (PCMLine::getVideoPixeBylCalc, pcmline.cpp:249-311)
    // Fused deinterleave (stc007_bulk_kernel<true>): the warp that decoded a frame keeps its line words in shared memory and
    // finishes, when the frame is complete, every data block whose eight lines lie inside the frame (the first 2*lpf - 112 of the
    // 2*lpf blocks that start in it; the blocks that reach into the next frame are left to stc007_deint_kernel).  Standard
    // setting only: 14 bit, parity check forced, P and Q correction, CRC respected, plain samples.
    i16 *samples; u8 *sflags;       // [blocks][6] each
    u32 *broken_bits; u8 *broken_sum;   // candidate bits of the countdown walk (zeroed before the launch; set with atomics)
    long long block0;               // block index of assembled line 0 of frame 0 of the records (lead-in lines in front of it)
    int lpf;                        // lines per field of the standard
};
enum { BULK_FUSE_HF = 288, BULK_FUSE_BYTES = 2*8*BULK_FUSE_HF*2+2*BULK_FUSE_HF };      // per warp: words of the frame's lines (word-major) + valid flags

// bits [off, off+len) of the MSB-first 128-bit stream B0:B1:B2:B3
template<int OFF, int LEN>
__device__ __forceinline__ u32 stream_field(u32 b0, u32 b1, u32 b2, u32 b3)
{
    constexpr int idx = OFF>>5, sh = 32-(OFF&31)-LEN;
    const u32 hi = (idx==0) ? b0 : ((idx==1) ? b1 : ((idx==2) ? b2 : b3));
    const u32 lo = (idx==0) ? b1 : ((idx==1) ? b2 : ((idx==2) ? b3 : 0u));
    constexpr u32 mask = (1u<<LEN)-1u;
    if constexpr (sh>=0) return (hi>>sh)&mask;
    else return __funnelshift_l(lo, hi, (u32)(-sh))&mask;
}

// bit_i = G_i | (E_i & bit_{i-1}) over the MSB-first stream (bit 0 = MSB of g[0]): carry chain of (G|E) + G on the
// bit-reversed vectors.
__device__ __forceinline__ void resolve_equal_cells(u32 *g, const u32 *ge)
{
    u32 gr[4], er[4];
#pragma unroll
    for(int i=0;i<4;i++) { gr[i] = __brev(g[i]); er[i] = __brev(ge[i]&~g[i]); }       // word i now holds line bits 32i..32i+31, LSB first
    u64 alo = ((u64)(gr[1]|er[1])<<32)|(gr[0]|er[0]), ahi = ((u64)(gr[3]|er[3])<<32)|(gr[2]|er[2]);
    u64 blo = ((u64)gr[1]<<32)|gr[0], bhi = ((u64)gr[3]<<32)|gr[2];
    u64 slo = alo+blo;
    u64 cy = (slo<alo) ? 1ull : 0ull;
    u64 shi = ahi+bhi+cy;
    u64 cout = ((shi<ahi)||(cy&&(shi==ahi))) ? 1ull : 0ull;
    u64 clo = slo^alo^blo, chi = shi^ahi^bhi;                   // carry into each bit
    u64 rlo = (clo>>1)|(chi<<63), rhi = (chi>>1)|(cout<<63);    // carry out of each bit = the decoded bit
    g[0] = __brev((u32)rlo); g[1] = __brev((u32)(rlo>>32)); g[2] = __brev((u32)rhi); g[3] = __brev((u32)(rhi>>32));
}

__device__ __forceinline__ bool packed_almost_silent(u32 w01, u32 w23, u32 w45)
{   // stc007line.cpp:582-606: at least two of the six samples in [-16, 15] after <<2, i.e. 14-bit word in {0..3, 0x3FFC..0x3FFF}
    const u32 a = ((w01+0x00040004u)&0x3FF83FF8u), b = ((w23+0x00040004u)&0x3FF83FF8u), c = ((w45+0x00040004u)&0x3FF83FF8u);
    const int cnt = ((a&0xFFFFu)==0)+((a>>16)==0)+((b&0xFFFFu)==0)+((b>>16)==0)+((c&0xFFFFu)==0)+((c>>16)==0);
    return cnt>=2;
}
__device__ __forceinline__ int packed_diff8(u32 a01, u32 a23, u32 a45, u32 a67, u32 b01, u32 b23, u32 b45, u32 b67)
{   // low 8 bits of each 16-bit word only (stc007line.cpp:329-356)
    const u32 m = 0x00FF00FFu;
    return __popc((a01^b01)&m)+__popc((a23^b23)&m)+__popc((a45^b45)&m)+__popc((a67^b67)&m);
}
__device__ __forceinline__ bool packed_control_block(u32 w01, u32 w23, u32 w45, u32 w67)
{
    return (w01==0x0CCC3333u)&&(w23==0x0CCC3333u)&&((w45&0xFFFFu)==0)&&(((w67>>16)&0x0FF0u)==0);
}

template<bool FUSE>
__global__ void __launch_bounds__(BULK_MAX_WARPS*32, 1) stc007_bulk_kernel(const __grid_constant__ BulkParams p)
{
    extern __shared__ __align__(128) u8 dsm[];
    u16 *crc_tab = (u16 *)(dsm+BULK_BAR_BYTES);                 // [3][256]: byte table, 7-byte advance of the low / high CRC byte
    const int warp = threadIdx.x>>5, lane = threadIdx.x&31;
    // fused deinterleave: this warp's line words of the current frame, word-major per field, and a valid flag per line
    u16 *fw = (u16 *)(dsm+BULK_SMEM_HEADER+(size_t)p.warps*BULK_STAGES*BULK_ROWS*p.slot_bytes+(size_t)warp*BULK_FUSE_BYTES);
    u8 *fok = (u8 *)(fw+2*8*BULK_FUSE_HF);
    for(int i=threadIdx.x;i<3*256;i+=blockDim.x) crc_tab[i] = c_crc8[i];
    BulkRing rb(dsm, BULK_SMEM_HEADER, p.luma, p.H, p.W, p.stride, p.f0, p.n_frames, p.use_tma, p.warps, p.slot_bytes);
    __syncthreads();
    rb.prime();

    // A step holds BULK_ROWS consecutive rows of the frame: rows alternate between the two fields, lane l holds field l&1,
    // line (l>>1) of the step.
    const int hf = p.H/2;
    const int ref = p.ref;
    const int fld = lane&1;

    u32 c01 = 0, c23 = 0, c45 = 0, c67 = 0;     // words of this field's last line in the previous step (duplicate check)
    bool c_cb = false;
    u32 frame_bad = 0;                          // bit 0 / 1: field 0 / 1 has a line this kernel cannot take
    const u32 rec5 = (u32)p.ref|((u32)p.black<<8)|((u32)p.white<<16);                // ref, black, white, hyst = 0
    const u32 rec6 = (u32)(u16)p.coords.start|((u32)(u16)p.coords.stop<<16);

    for(long long it=0;it<rb.n_items;it++)
    {
        const BulkItem t = rb.item(it);
        const int f = t.f, b = t.b, r0 = t.r0, rows = t.rows;
        const int k = (r0>>1)+(lane>>1);                        // line of the field
        const bool active = lane<rows;
        const u8 *row = rb.acquire(t)+(size_t)lane*p.slot_bytes;
        // ---- 128 bit cells of this lane's row
        u32 g[4], ge[4];
#pragma unroll
        for(int w=0;w<4;w++)
        {
            u32 a = 0, c = 0;
#pragma unroll
            for(int j=0;j<32;j++)
            {
                const int v = row[p.pos[32*w+j]];
                a = __funnelshift_l((u32)(ref-v), a, 1);        // pixel >  ref
                c = __funnelshift_l((u32)(ref-1-v), c, 1);      // pixel >= ref
            }
            g[w] = a; ge[w] = c;
        }
        rb.release(it);
        const bool any_eq = ((ge[0]^g[0])|(ge[1]^g[1])|(ge[2]^g[2])|(ge[3]^g[3]))!=0;
        if(__any_sync(0xFFFFFFFFu, any_eq)) resolve_equal_cells(g, ge);
        // ---- words and CRCC (two independent table chains over the two halves of the 14-byte message)
        const u32 w0 = stream_field<0, 14>(g[0], g[1], g[2], g[3]), w1 = stream_field<14, 14>(g[0], g[1], g[2], g[3]);
        const u32 w2 = stream_field<28, 14>(g[0], g[1], g[2], g[3]), w3 = stream_field<42, 14>(g[0], g[1], g[2], g[3]);
        const u32 w4 = stream_field<56, 14>(g[0], g[1], g[2], g[3]), w5 = stream_field<70, 14>(g[0], g[1], g[2], g[3]);
        const u32 w6 = stream_field<84, 14>(g[0], g[1], g[2], g[3]), w7 = stream_field<98, 14>(g[0], g[1], g[2], g[3]);
        u32 w8 = g[3]&0xFFFFu;
        u32 crc_a = 0xFFFFu, crc_b = 0;
#pragma unroll
        for(int j=0;j<7;j++)
        {
            const u32 ma = (g[j>>2]>>(24-8*(j&3)))&0xFFu, mb = (g[(j+7)>>2]>>(24-8*((j+7)&3)))&0xFFu;
            crc_a = ((crc_a<<8)^crc_tab[((crc_a>>8)^ma)&0xFFu])&0xFFFFu;
            crc_b = ((crc_b<<8)^crc_tab[((crc_b>>8)^mb)&0xFFu])&0xFFFFu;
        }
        const u32 crc = (u32)crc_tab[256+(crc_a&0xFFu)]^(u32)crc_tab[512+(crc_a>>8)]^crc_b;
        const bool crc_ok = (crc==w8);
        u32 w01 = w0|(w1<<16), w23 = w2|(w3<<16), w45 = w4|(w5<<16), w67 = w6|(w7<<16);
        const bool is_cb = crc_ok&&packed_control_block(w01, w23, w45, w67);
        {
            const u32 bad = __ballot_sync(0xFFFFFFFFu, active&&((!crc_ok)||(is_cb&&(k!=0))));
            if(bad&0x55555555u) frame_bad |= 1u;
            if(bad&0xAAAAAAAAu) frame_bad |= 2u;
        }
        // ---- VideoToDigital per-field rules for a valid line; the previous line of the same field sits two lanes down
        u32 p01 = __shfl_up_sync(0xFFFFFFFFu, w01, 2), p23 = __shfl_up_sync(0xFFFFFFFFu, w23, 2);
        u32 p45 = __shfl_up_sync(0xFFFFFFFFu, w45, 2), p67 = __shfl_up_sync(0xFFFFFFFFu, w67, 2);
        bool p_cb = __shfl_up_sync(0xFFFFFFFFu, is_cb ? 1 : 0, 2)!=0;
        if(lane<2) { p01 = c01; p23 = c23; p45 = c45; p67 = c67; p_cb = c_cb; }
        if((k==0)||p_cb) { p01 = p23 = p45 = p67 = 0; }         // field start / Control Block before: last_line is a cleared line
        bool silent;
        if(p.line_dup&2)
        {   // M2 tape: the range/sign expansion decides what is near silence
            u16 t6[6] = { (u16)(w01&0xFFFFu), (u16)(w01>>16), (u16)(w23&0xFFFFu), (u16)(w23>>16), (u16)(w45&0xFFFFu), (u16)(w45>>16) };
            silent = words_almost_silent(t6, true);
        }
        else silent = packed_almost_silent(w01, w23, w45);
        bool forced_bad = false;
        if((p.line_dup&1)&&!is_cb)
        {
            if(k==0) forced_bad = FINE_FIRST_LINE_DUP;           // first PCM line of the field, no Control Block before it (en_first_line_dup)
            else forced_bad = (packed_diff8(w01, w23, w45, w67, p01, p23, p45, p67)<=(BITS_PCM_DATA/32))&&!silent;
        }
        const int last = rows-2+fld;                            // this field's last row of the step (rows is even)
        c01 = __shfl_sync(0xFFFFFFFFu, w01, last); c23 = __shfl_sync(0xFFFFFFFFu, w23, last);
        c45 = __shfl_sync(0xFFFFFFFFu, w45, last); c67 = __shfl_sync(0xFFFFFFFFu, w67, last);
        c_cb = __shfl_sync(0xFFFFFFFFu, is_cb ? 1 : 0, last)!=0;
        // ---- record
        u32 flags, r5 = rec5, r6 = rec6, r7 = 0;
        bool silent_out = silent;
        if(is_cb)
        {   // STC007Line::setServCtrlBlk: words 4..7 survive, CRCC recomputed, everything else cleared
            w01 = 0; w23 = 0;
            u16 t[8] = { 0, 0, 0, 0, (u16)(w45&0xFFFFu), (u16)(w45>>16), (u16)(w67&0xFFFFu), (u16)(w67>>16) };
            w8 = crc_stc007(t);
            flags = SDV_LF_CRC_OK|SDV_LF_CRC_OK_IGN;
            r5 = 0; r6 = (u32)(u16)NO_COORD_LEFT|((u32)(u16)NO_COORD_RIGHT<<16); r7 = (u32)SDV_SRV_CTRL_BLOCK<<8;
            silent_out = packed_almost_silent(w01, w23, w45);
        }
        else
        {
            flags = SDV_LF_CRC_OK_IGN|SDV_LF_BW_SET|SDV_LF_BY_EXT;
            flags |= forced_bad ? SDV_LF_FORCED_BAD : SDV_LF_CRC_OK;
        }
        if(silent_out) flags |= SDV_LF_ALMOST_SILENT;
        if(active)
        {
            const size_t ridx = (size_t)f*p.H+(size_t)fld*hf+k;
            uint4 *dst = (uint4 *)(p.recs+ridx);
            dst[0] = make_uint4(w01, w23, w45, w67);
            dst[1] = make_uint4(w8|(flags<<16), r5, r6, r7);
            if(p.aux)
            {   // ref_low, ref_high, marker_start_bg | marker_start_ed, marker_stop_ed | word_crc_mask, word_valid_mask | pad
                const u32 masks = (is_cb||forced_bad) ? 0u : 0x01FF01FFu;
                *(uint4 *)(p.aux+ridx) = make_uint4(is_cb ? 0u : ((u32)p.ref|((u32)p.ref<<8)), 0u, masks, 0u);
            }
        }
        if(FUSE)
        {
            if(active)
            {
                u16 *d = fw+(size_t)fld*8*BULK_FUSE_HF+k;
                d[0*BULK_FUSE_HF] = (u16)w01; d[1*BULK_FUSE_HF] = (u16)(w01>>16); d[2*BULK_FUSE_HF] = (u16)w23; d[3*BULK_FUSE_HF] = (u16)(w23>>16);
                d[4*BULK_FUSE_HF] = (u16)w45; d[5*BULK_FUSE_HF] = (u16)(w45>>16); d[6*BULK_FUSE_HF] = (u16)w67; d[7*BULK_FUSE_HF] = (u16)(w67>>16);
                fok[fld*BULK_FUSE_HF+k] = ((flags&SDV_LF_CRC_OK)&&!is_cb) ? 1 : 0;      // line_rec_ok: a service line gives no trusted words
            }
            if(b==rb.nbatch-1)
            {   // every block of this frame whose lines all lie inside it: assembled line a = field 0 lines, lpf - hf empty lines,
                // field 1 lines, empty lines; block a takes word j of line a + 16 j
                __syncwarp();
                const int lpf = p.lpf, n_in = 2*lpf-112;
                const long long bf = p.block0+(long long)f*2*lpf;
                for(int a=lane;a<n_in;a+=32)
                {
                    BlockIn in; in.ok = 0;
#pragma unroll
                    for(int j=0;j<8;j++)
                    {
                        int L = a+16*j, q = 0;
                        if(L>=lpf) { L -= lpf; q = 1; }
                        u16 wv = 0; u32 okv = 0;
                        if(L<hf) { wv = fw[(size_t)q*8*BULK_FUSE_HF+(size_t)j*BULK_FUSE_HF+L]; okv = fok[q*BULK_FUSE_HF+L]; }
                        in.w[j] = wv; in.sw[j] = 0;
                        in.ok |= (u8)(okv<<j);
                    }
                    Block blk;
                    deint_block_std14(&blk, &in);
                    blk.m2 = 0;
                    const long long bi = bf+a;
                    u32 f03, f45;
                    blk_output_flags(&blk, &f03, &f45);
                    u32 *ds = (u32 *)(p.samples+bi*6);
                    ds[0] = (((u32)blk.words[0]<<2)&0xFFFFu)|((u32)blk.words[1]<<18);
                    ds[1] = (((u32)blk.words[2]<<2)&0xFFFFu)|((u32)blk.words[3]<<18);
                    ds[2] = (((u32)blk.words[4]<<2)&0xFFFFu)|((u32)blk.words[5]<<18);
                    u16 *df = (u16 *)(p.sflags+bi*6);
                    df[0] = (u16)f03; df[1] = (u16)(f03>>16); df[2] = (u16)f45;
                    if((blk.audio_state==SDV_AUD_BROKEN)&&!blk_silent(&blk)&&p.broken_bits)
                    {
                        atomicOr(&p.broken_bits[bi>>5], 1u<<(u32)(bi&31));
                        p.broken_sum[bi>>10] = 1;
                    }
                }
                __syncwarp();
            }
        }
        if(b==rb.nbatch-1)
        {   // frame done
            if(lane<2) p.clean[2*(size_t)f+lane] = ((frame_bad>>lane)&1u) ? 0 : 1;
            if((lane==0)&&frame_bad) atomicMin(p.first_unclean, f);
            frame_bad = 0; c01 = c23 = c45 = c67 = 0; c_cb = false;
        }
    }
}

}   // namespace sdv
