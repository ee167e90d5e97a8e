// bulk_ring.cuh -- how luma rows reach shared memory in the bulk line-decode kernels (stc007_bulk_kernel,
// pcm1_bulk_kernel, pcm16x0_bulk_kernel): the per-warp staging ring and its host launch plan.
//
// Persistent grid, work unit = one frame, frames dealt round-robin over every warp of the grid.  A warp walks its frames
// in items of BULK_ROWS consecutive rows (the last item of a frame may be shorter; both fields interleaved).  Each warp
// owns a ring of BULK_STAGES stages in dynamic shared memory.  With a 16-byte aligned luma pointer and row pitch the
// rows of an item arrive in ONE 1-D bulk copy (they are contiguous in memory: rows*stride bytes), completed on the
// stage's mbarrier; otherwise the warp fills the stage with plain loads when it acquires it.
//
// Dynamic shared memory of a block: [0, BULK_BAR_BYTES) the ring barriers, [BULK_BAR_BYTES, header) the kernel's own
// tables, then the rings of all warps (warps x BULK_STAGES x BULK_ROWS x slot_bytes), then whatever the kernel keeps per
// warp behind them.
//
// Slot contract: row r of an item is at stage + r*slot_bytes, and its bytes [0, W) are valid from acquire() until
// release().  With bulk copies slot_bytes is the row pitch (the padding comes along); otherwise it is the compact slot,
// the smallest odd number of 16-byte units that holds W bytes (fewest bank conflicts between the 32 rows a warp reads
// together).
#pragma once
#include "sdv_common.cuh"

namespace sdv {

enum { BULK_MAX_WARPS = 4, BULK_STAGES = 2, BULK_ROWS = 32, BULK_BAR_BYTES = 128 };
static_assert(BULK_MAX_WARPS*BULK_STAGES*8<=BULK_BAR_BYTES, "ring barriers do not fit their area");

__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(u64 *bar, u32 bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity)
{
    u32 done;
    do
    {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    }
    while(!done);
}
__device__ __forceinline__ void bulk_g2s(u32 dst_smem, const void *src, u32 bytes, u64 *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst_smem), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

struct BulkItem
{
    int f, b, r0, rows;             // frame, step of the frame, its first row and row count
    int s; u32 parity;              // ring stage and the phase of its barrier that completes this item
};

// One warp's ring.  Construct it in every thread of the block before the __syncthreads() that publishes the kernel's
// header tables (it initialises the barriers), then prime() it.  Per item it: acquire(item(it)), read the rows,
// release(it) -- after which the stage may be overwritten.
struct BulkRing
{
    const u8 *luma; size_t stride; int H, W, f0;
    int use_tma, lane, nbatch; u32 slot_bytes, stage_bytes;
    u8 *ring; u64 *bar;
    long long gw, gstride, n_items;

    // frames [f0, f0+n_frames) of luma; header = first byte of the rings in dsm
    __device__ __forceinline__ BulkRing(u8 *dsm, u32 header, const u8 *luma_, int H_, int W_, size_t stride_, int f0_,
                                        int n_frames, int use_tma_, int warps, u32 slot_bytes_)
        : luma(luma_), stride(stride_), H(H_), W(W_), f0(f0_), use_tma(use_tma_), lane(threadIdx.x&31), slot_bytes(slot_bytes_)
    {
        const int warp = threadIdx.x>>5;
        stage_bytes = BULK_ROWS*slot_bytes;
        ring = dsm+header+(size_t)warp*BULK_STAGES*stage_bytes;
        bar = (u64 *)dsm+warp*BULK_STAGES;
        if(use_tma&&(lane==0))
        {
            for(int s=0;s<BULK_STAGES;s++) mbar_init(&bar[s], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        nbatch = (H+BULK_ROWS-1)/BULK_ROWS;
        gw = (long long)blockIdx.x*warps+warp; gstride = (long long)gridDim.x*warps;
        const long long my_units = (gw<n_frames) ? ((n_frames-gw+gstride-1)/gstride) : 0;
        n_items = my_units*nbatch;
    }

    __device__ __forceinline__ BulkItem item(long long it) const
    {
        BulkItem t;
        t.f = f0+(int)(gw+(it/nbatch)*gstride);
        t.b = (int)(it%nbatch); t.r0 = t.b*BULK_ROWS;
        t.rows = (H-t.r0<BULK_ROWS) ? (H-t.r0) : BULK_ROWS;
        t.s = (int)((unsigned long long)it%BULK_STAGES);
        t.parity = (u32)(((unsigned long long)it/BULK_STAGES)&1);
        return t;
    }

    __device__ __forceinline__ void issue(long long it) const
    {
        const BulkItem t = item(it);
        if(lane==0)
        {
            const u32 bytes = (u32)t.rows*(u32)stride;
            mbar_expect_tx(&bar[t.s], bytes);
            bulk_g2s(smem_u32(ring)+(u32)t.s*stage_bytes, luma+((size_t)t.f*H+(size_t)t.r0)*stride, bytes, &bar[t.s]);
        }
        __syncwarp();
    }

    __device__ __forceinline__ void prime() const
    {
        if(use_tma)
        {
#pragma unroll
            for(int i=0;i<BULK_STAGES;i++) if(n_items>i) issue(i);
        }
    }

    // base of the item's stage once its rows are there
    __device__ __forceinline__ u8 *acquire(const BulkItem &t) const
    {
        u8 *stage = ring+(size_t)t.s*stage_bytes;
        if(use_tma) mbar_wait(&bar[t.s], t.parity);
        else
        {
            __syncwarp();
            for(int r=0;r<t.rows;r++)
            {
                const u8 *src = luma+((size_t)t.f*H+(size_t)(t.r0+r))*stride;
                u8 *dst = stage+(size_t)r*slot_bytes;
                for(int j=lane;j<W;j+=32) dst[j] = __ldg(src+j);
            }
            __syncwarp();
        }
        return stage;
    }

    // every lane is done with item it's rows: the stage takes item it+BULK_STAGES
    __device__ __forceinline__ void release(long long it) const
    {
        __syncwarp();
        if(use_tma&&(it+BULK_STAGES<n_items)) issue(it+BULK_STAGES);
    }
};

// Launch plan of a bulk kernel with [header] bytes of shared memory in front of the rings.
struct BulkPlan
{
    int use_tma; u32 slot_bytes;
    int warps;                      // < 1: not even one warp fits
    size_t smem;                    // dynamic shared memory of a block
};

// Count the warps of [pl]'s slot layout with [extra] bytes per warp behind the rings.
inline BulkPlan bulk_plan_warps(BulkPlan pl, size_t header, size_t extra)
{
    const size_t per_warp = (size_t)BULK_STAGES*BULK_ROWS*pl.slot_bytes+extra;
    pl.warps = (int)((size_t)(227*1024-header)/per_warp);
    if(pl.warps>BULK_MAX_WARPS) pl.warps = BULK_MAX_WARPS;
    pl.smem = header+(size_t)pl.warps*per_warp;
    return pl;
}

inline BulkPlan bulk_plan(int W, int stride, const void *luma, size_t header)
{
    const u32 copy_bytes = (u32)((W+15)&~15);
    const u32 compact = ((copy_bytes/16)&1) ? copy_bytes : (copy_bytes+16);
    BulkPlan pl;
    pl.use_tma = (((size_t)stride%16)==0)&&((((uintptr_t)luma)%16)==0);
    pl.slot_bytes = pl.use_tma ? (u32)stride : compact;
    pl = bulk_plan_warps(pl, header, 0);
    if((pl.warps<1)&&pl.use_tma)
    {   // very wide pitch: the compact layout
        pl.use_tma = 0; pl.slot_bytes = compact;
        pl = bulk_plan_warps(pl, header, 0);
    }
    return pl;
}

}   // namespace sdv
