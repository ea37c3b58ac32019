/*
 * dpf_kernels.cu -- sm_100a kernels of the DPF evaluation engine.
 *
 * One kernel does the whole hot path of the reference's dpf_hybrid_kernel
 * (dpf_gpu/dpf/dpf_hybrid.cu:38-256): GGM-tree expansion of every key over the
 * full domain, fused with the inner product against the table, plus the
 * reduction -- but organised for Blackwell rather than translated:
 *
 *   work item   = (group of 32 keys) x (one 2^s-leaf subtree).  A warp owns a
 *                 work item; LANE = KEY.  All 32 lanes walk the same tree shape,
 *                 so control flow is warp-uniform and every table row a warp
 *                 needs is ONE broadcast 128-bit load shared by 32 keys (the
 *                 reference re-reads the table once per key).  For batches
 *                 smaller than a warp the mapping generalises to lane = (key,
 *                 subtree slot): kpw keys x 32/kpw adjacent subtrees per warp, so a
 *                 single query still uses every lane (the role the reference gives
 *                 to dpf_coop.cu).
 *   expansion   = per-thread depth-first search: a node's two children are
 *                 produced together in registers (shared AES key schedule /
 *                 shared first-round quarter rounds), the right child parks in a
 *                 per-thread shared-memory slot (one slot per tree height), the
 *                 left child is descended into.  No global scratch, no
 *                 __syncthreads in the main loop (the reference ping-pongs two
 *                 global stacks with two barriers per step).
 *   MAC         = only the low 32 bits of a leaf survive (dpf_wrapper.cu:182),
 *                 so the product is 32-bit IMADs against an int32 table stored
 *                 in breadth-first leaf order (4x less table traffic than the
 *                 reference's 128-bit table, ~20x fewer MAC instructions).  With
 *                 4+ keys per warp the 4 lanes of a quad split the row into 4
 *                 column slices and trade their leaves by shuffle (DevEnv, QUAD).
 *   corrections = the 32 keys' correction words live in shared memory, laid out
 *                 [level][bank][bit][key] so a warp's 16-byte reads are
 *                 conflict free.
 *   AES         = T-table AES with the four tables replicated per bank in
 *                 shared memory (4 x 32 KiB): lane L only ever touches bank L,
 *                 so lookups are conflict-free, and the shared address of a
 *                 lookup is formed by ONE PRMT (byte insert into a 64 KiB-aligned
 *                 base) + the LDS immediate offset.
 *   frontier    = the top of every key's tree is expanded once and the seeds of all
 *                 depth-F nodes stored; work items then start from their frontier
 *                 node instead of re-walking from the root, so items can be small
 *                 (good load balance) without paying a root-to-subtree walk each.
 *   one launch  = a whole evaluation is ONE cooperative launch: phase `top` clears the
 *                 result and the ticket counters and builds the frontier, a grid-wide
 *                 barrier follows, phase `main` does the work and block 0 re-arms the
 *                 top-phase tickets for the next launch.  (The reference's step is
 *                 cudaMemcpy + kernel + cudaMemcpy with a stream created per call,
 *                 dpf_wrapper.cu:150-176; ours was memset, memset, kernel, kernel.)
 *   wide rows   = NV uint4 of a table row per pass (16/32/64 int32 columns), loaded
 *                 before the leaf expansion: a lane's NV/4 uint4 slice of both rows
 *                 (quad layout), or the first 64 bytes of both rows with the rest
 *                 streamed chunk by chunk during the MAC (1 or 2 keys per warp).
 *   scheduling  = persistent blocks; warps draw subtrees from a per-key-group
 *                 ticket counter (atomicAdd), blocks migrate to the next key
 *                 group when theirs runs dry, partial sums leave through
 *                 red.global.add.u32.
 */
#include "dpf_kernels.cuh"

#include <algorithm>
#include <atomic>

#include "dpf_core.cuh"

namespace b200dpf {

namespace {

__constant__ uint32_t c_te0[256];

/* ---- AES table policy on the device -------------------------------------- */
struct AesSmemTables {
    /* shared-window address of (table region + lane*4); the region base is a
     * multiple of 64 KiB, so byte 1 of this value is zero. */
    uint32_t lanebase;

    template <int K, int BYTE>
    __device__ __forceinline__ uint32_t te(uint32_t word) const
    {
        /* address = lanebase with byte 1 replaced by the index byte:
         * entry v of table K for lane L sits at v*256 + (K&1)*128 + (K>>1)*65536 + L*4 */
        const uint32_t addr = __byte_perm(word, lanebase, 0x7604u | (BYTE << 4));
        uint32_t v;
        asm("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"((K & 1) * 128 + (K >> 1) * 65536));
        return v;
    }
};

struct NoTables {
    template <int K, int BYTE>
    __device__ __forceinline__ uint32_t te(uint32_t) const { return 0; }
};

template <int PRF> struct TablePolicy { typedef NoTables type; };
template <> struct TablePolicy<PRF_AES128> { typedef AesSmemTables type; };

/* ---- cp.async.bulk (TMA) + mbarrier primitives ----------------------------- */
namespace tma {

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; spin++) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (spin > (1u << 28)) __trap();   /* a lost arrival must not hang the GPU */
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

}  // namespace tma

/* ---- per-thread environment for the shared traversal code ---------------- */
/*
 * Two layouts of the inner product (MAC):
 *   QUAD = false  every lane multiplies its own key's leaves against the whole row: it loads
 *                 all NV uint4 of both rows of a leaf pair (the per-lane layout; the only one
 *                 possible with 1 or 2 keys per warp, where no two lanes share a subtree);
 *   QUAD = true   (keys per warp >= 4) the 4 lanes of a quad hold 4 keys of the same subtree,
 *                 and quad lane j owns the column slice {uint4 j, j+4, j+8, ...}: it loads
 *                 NV/4 uint4 of each row, takes its partners' leaves with 6 shuffles, and
 *                 accumulates 4 keys x its columns.  Same IMAD count, 4x fewer row bytes
 *                 through the LSU per leaf pair (a broadcast LDG.128 still costs 4 wavefronts).
 *                 acc[16*c + 4*m + e] is key (kslot ^ m), column 4*(4c + j) + e.
 */
template <int PRF, int NV, int THREADS, int MODE, bool QUAD>
struct DevEnv {
    static constexpr int ROW_V = QUAD ? NV / 4 : 4;   /* uint4 of each row held in registers */
    typename TablePolicy<PRF>::type ta;
    const uint4 *cw_lane;       /* &cw_s[lane]; entry (level,bank,bit) at +((level*2+bank)*2+bit)*32 */
    const uint32_t *cwlo_lane;  /* &cwlo_s[lane]; entry (bank,bit) at +(bank*2+bit)*32 */
    uint4 *stack_lo, *stack_hi; /* pre-offset by tid; level l at +l*THREADS */
    int stack_split;
    const uint4 *rows;          /* first row of the current subtree, at this pass's column */
    uint32_t row_stride_v;
    uint32_t qlane;             /* QUAD: lane & 3, the column slice this lane owns */
    uint32_t acc[4 * NV];
    uint4 ra[ROW_V], rb[ROW_V]; /* prefetched row data of a leaf pair: QUAD, this lane's slice of both
                                 * rows; otherwise the first 64 bytes of both */
    uint32_t *leaf_out;         /* leaf cache slot of the subtree's first leaf for this lane, or null */
    uint4 *front_out;           /* MODE_FRONTIER: &frontier[(kg*nfront + first node)*kpw + key slot] */
    uint32_t kpw;               /* keys per warp */
    /* expand mode */
    uint32_t *share_row;        /* shares + key*n */
    uint32_t pos_base;          /* global leaf position of the subtree's first leaf */
    int depth;
    bool key_valid;

    __device__ __forceinline__ Seed cw(int level, uint32_t bank, uint32_t bit) const
    {
        const uint4 v = cw_lane[((level * 2 + (int)bank) * 2 + (int)bit) * 32];
        return make_seed(v.x, v.y, v.z, v.w);
    }
    __device__ __forceinline__ uint32_t cw_lo(uint32_t bank, uint32_t bit) const
    {
        return cwlo_lane[(bank * 2 + bit) * 32];
    }
    __device__ __forceinline__ uint4 *slot(int h) const
    {
        const int l = h - 1;
        return (l < stack_split ? stack_lo : stack_hi) + l * THREADS;
    }
    __device__ __forceinline__ void push(int h, const Seed &s) const
    {
        *slot(h) = make_uint4(s.x, s.y, s.z, s.w);
    }
    __device__ __forceinline__ Seed pop(int h) const
    {
        const uint4 v = *slot(h);
        return make_seed(v.x, v.y, v.z, v.w);
    }
    static constexpr bool MAC = (MODE == MODE_FUSED || MODE == MODE_GROUPED || MODE == MODE_FUSED_TMA);   /* leaves feed the inner product */
    static constexpr bool STAGED = (MODE == MODE_FUSED_TMA);
    /* STAGED: the work item's 2^s rows were requested with one cp.async.bulk when the item was drawn;
     * they are first needed s-1 node expansions later, which hides the copy */
    const uint4 *tile;          /* this warp's staged rows (shared memory) */
    uint32_t tile_bar;          /* shared-window address of this warp's mbarrier */
    uint32_t tile_phase;
    bool tile_pending;

    __device__ __forceinline__ void leaf_prefetch(uint32_t local_pos)
    {
        if constexpr (STAGED) {
            if (tile_pending) {
                tma::mbar_wait(tile_bar, tile_phase);
                tile_phase ^= 1u;
                tile_pending = false;
            }
            const uint4 *r = tile + (size_t)local_pos * 4;   /* 64-byte rows: NV = 4 */
            if constexpr (QUAD) {
                ra[0] = r[qlane];
                rb[0] = r[4 + qlane];
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) ra[j] = r[j];
#pragma unroll
                for (int j = 0; j < 4; j++) rb[j] = r[4 + j];
            }
        } else if constexpr (MAC) {
            if constexpr (QUAD) {
                const uint4 *r = rows + (size_t)local_pos * row_stride_v + qlane;
#pragma unroll
                for (int c = 0; c < ROW_V; c++) ra[c] = __ldg(r + 4 * c);
#pragma unroll
                for (int c = 0; c < ROW_V; c++) rb[c] = __ldg(r + row_stride_v + 4 * c);
            } else {
                const uint4 *r = rows + (size_t)local_pos * row_stride_v;
#pragma unroll
                for (int j = 0; j < 4; j++) ra[j] = __ldg(r + j);
#pragma unroll
                for (int j = 0; j < 4; j++) rb[j] = __ldg(r + row_stride_v + j);
            }
        }
    }
    __device__ __forceinline__ void leaf_pair(uint32_t local_pos, uint32_t v0, uint32_t v1)
    {
        if constexpr (MAC) {
            if (leaf_out != nullptr) {   /* coalesced: 32 keys x 4 bytes per leaf */
                leaf_out[(size_t)local_pos * 32] = v0;
                leaf_out[(size_t)(local_pos + 1) * 32] = v1;
            }
            if constexpr (QUAD) {
                /* slot m: the leaves of key kslot ^ m, held by quad lane qlane ^ m */
                uint32_t w0[4], w1[4];
                w0[0] = v0;
                w1[0] = v1;
#pragma unroll
                for (int m = 1; m < 4; m++) {
                    w0[m] = __shfl_xor_sync(0xffffffffu, v0, m);
                    w1[m] = __shfl_xor_sync(0xffffffffu, v1, m);
                }
#pragma unroll
                for (int c = 0; c < ROW_V; c++) {
#pragma unroll
                    for (int m = 0; m < 4; m++) {
                        acc[16 * c + 4 * m + 0] += w0[m] * ra[c].x + w1[m] * rb[c].x;
                        acc[16 * c + 4 * m + 1] += w0[m] * ra[c].y + w1[m] * rb[c].y;
                        acc[16 * c + 4 * m + 2] += w0[m] * ra[c].z + w1[m] * rb[c].z;
                        acc[16 * c + 4 * m + 3] += w0[m] * ra[c].w + w1[m] * rb[c].w;
                    }
                }
            } else {
                const uint4 *r = rows + (size_t)local_pos * row_stride_v;
#pragma unroll
                for (int c = 0; c < NV / 4; c++) {
                    uint4 na[4], nb[4];
                    if (c + 1 < NV / 4) {   /* next 64 bytes of both rows while this chunk is multiplied */
#pragma unroll
                        for (int j = 0; j < 4; j++) na[j] = __ldg(r + 4 * (c + 1) + j);
#pragma unroll
                        for (int j = 0; j < 4; j++) nb[j] = __ldg(r + row_stride_v + 4 * (c + 1) + j);
                    }
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        acc[16 * c + 4 * j + 0] += v0 * ra[j].x + v1 * rb[j].x;
                        acc[16 * c + 4 * j + 1] += v0 * ra[j].y + v1 * rb[j].y;
                        acc[16 * c + 4 * j + 2] += v0 * ra[j].z + v1 * rb[j].z;
                        acc[16 * c + 4 * j + 3] += v0 * ra[j].w + v1 * rb[j].w;
                    }
                    if (c + 1 < NV / 4) {
#pragma unroll
                        for (int j = 0; j < 4; j++) { ra[j] = na[j]; rb[j] = nb[j]; }
                    }
                }
            }
        } else if (MODE == MODE_EXPAND && key_valid) {
            /* leaf position p holds index bitrev_depth(p) */
            const uint32_t p = pos_base + local_pos;
            share_row[__brev(p) >> (32 - depth)] = v0;
            share_row[__brev(p + 1) >> (32 - depth)] = v1;
        }
    }
    /* MODE_FRONTIER: whole seeds of two adjacent frontier nodes */
    __device__ __forceinline__ void node_pair(uint32_t local_pos, const Seed &c0, const Seed &c1)
    {
        front_out[(size_t)local_pos * kpw] = make_uint4(c0.x, c0.y, c0.z, c0.w);
        front_out[(size_t)(local_pos + 1) * kpw] = make_uint4(c1.x, c1.y, c1.z, c1.w);
    }
};

/* Block shape per (PRF, NV).  AES needs 128 KiB of the SM's shared memory for its
 * tables, so one block per SM; accumulators (4*NV registers) decide how many
 * threads fit the register file. */
template <int PRF, int NV> struct KernelShape { enum { THREADS = (NV <= 8 ? 256 : 384), MIN_BLOCKS = (NV <= 8 ? 2 : 1) }; };
#ifndef DPF_AES_THREADS
#define DPF_AES_THREADS 384      /* 8 warps (256) measured against 12 (384): profiles/r2_aes_block_size_ab.txt */
#endif
template <int NV> struct KernelShape<PRF_AES128, NV> { enum { THREADS = (NV <= 8 ? DPF_AES_THREADS : 256), MIN_BLOCKS = 1 }; };

extern __shared__ __align__(16) unsigned char g_dyn_smem[];

/* Grid-wide barrier of a cooperative launch (every block is resident, so spinning cannot
 * deadlock).  `bar` only ever counts up; `target` is the value it has once every block of THIS
 * launch has arrived (the host keeps the running total), compared wrap-safe. */
__device__ __forceinline__ void grid_barrier(uint32_t *bar, uint32_t target)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(bar, 1u);
        for (uint32_t spin = 0;; spin++) {
            uint32_t v;
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
            if ((int32_t)(v - target) >= 0) break;
            if (spin > (1u << 25)) __trap();   /* a lost arrival must not hang the GPU */
            __nanosleep(40);
        }
        __threadfence();
    }
    __syncthreads();
}

/* One traversal phase of a launch: every block walks the key groups (starting at its own offset so
 * blocks spread over groups), loads a group's correction words into shared memory when the group
 * still has tickets, and its warps draw work items until the group runs dry. */
__device__ __forceinline__ unsigned long long global_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

/* `quota`: tickets this WARP may draw in this call over all key groups (0xffffffff = no limit).
 * QUAD: the MAC layout of DevEnv; needs at least 4 keys per warp. */
template <int PRF, int NV, int THREADS, int MODE, bool QUAD = false>
__device__ __forceinline__ void run_phase(const EvalParams &p, const PhaseParams &ph,
                                          const typename TablePolicy<PRF>::type &ta, uint32_t quota = 0xffffffffu)
{
    const int tid = threadIdx.x;
    const int lane = tid & 31;

    uint4 *cw_s = reinterpret_cast<uint4 *>(g_dyn_smem + p.off_cw);
    uint32_t *cwlo_s = reinterpret_cast<uint32_t *>(g_dyn_smem + p.off_cwlo);
    uint4 *root_s = reinterpret_cast<uint4 *>(g_dyn_smem + p.off_root);
    volatile int *flag_s = reinterpret_cast<volatile int *>(g_dyn_smem + p.off_flag);

    /* lane -> (key slot within the group, subtree slot within the ticket) */
    const int kpw = 1 << p.kpw_log2;
    const int spw_log2 = 5 - p.kpw_log2;
    const int kslot = lane & (kpw - 1);
    const uint32_t sslot = (uint32_t)lane >> p.kpw_log2;
    const uint32_t ntickets = ph.nsub >> spw_log2;

    DevEnv<PRF, NV, THREADS, MODE, QUAD> env;
    env.ta = ta;
    env.qlane = (uint32_t)lane & 3u;
    env.cw_lane = cw_s + kslot;
    env.cwlo_lane = cwlo_s + kslot;
    env.kpw = (uint32_t)kpw;
    env.stack_lo = reinterpret_cast<uint4 *>(g_dyn_smem + p.off_stack_lo) + tid;
    env.stack_hi = reinterpret_cast<uint4 *>(g_dyn_smem + p.off_stack_hi) + tid - ph.stack_split * THREADS;
    env.stack_split = ph.stack_split;
    env.row_stride_v = p.row_stride_v;
    env.depth = p.depth;
    if constexpr (MODE == MODE_FUSED_TMA) {
        const int w = tid >> 5;
        env.tile = reinterpret_cast<const uint4 *>(g_dyn_smem + p.off_tile + ((size_t)w << (ph.s + 6)));
        env.tile_bar = (uint32_t)__cvta_generic_to_shared(g_dyn_smem + p.off_tile_bar + 8 * w);
        env.tile_phase = 0;
        env.tile_pending = false;
        if (lane == 0) {
            tma::mbar_init(env.tile_bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
    }

    constexpr bool GROUPED = (MODE == MODE_GROUPED);
    uint32_t taken = 0;
    for (int j = 0; j < p.key_groups; j++) {
        const int kg = (int)((blockIdx.x + (unsigned)j) % (unsigned)p.key_groups);

        /* what this key group evaluates: the context's one table, or (grouped) its own bin */
        int g_depth = p.depth, g_s = ph.s, g_walk_first = ph.walk_first_level, g_walk_steps = ph.walk_steps;
        int g_key_first = kg * kpw, g_key_last = p.nkeys - 1;
        uint32_t g_tickets = ntickets;
        const uint4 *g_table = p.table;
        if (GROUPED) {
            const GroupDesc g = p.groups[kg];
            g_depth = g.depth;
            g_s = g.s;
            g_walk_first = g.depth - 1;
            g_walk_steps = g.depth - g.s;
            g_key_first = (int)g.key_first;
            g_key_last = (int)(g.key_first + g.nkeys) - 1;
            g_tickets = g.nsub;
            g_table = p.table + g.table_off_v;
        }

        if (quota != 0xffffffffu && __syncthreads_and(taken >= quota)) break;   /* the block's share is done */
        if (tid == 0) *flag_s = (*reinterpret_cast<volatile uint32_t *>(ph.counters + kg) < g_tickets) ? 1 : 0;
        __syncthreads();
        const bool has_work = (*flag_s != 0);
        if (has_work) {
            /* correction words of this key group -> shared, [level][bank][bit][key] */
            const int per_key = g_depth * 4;
            for (int i = tid; i < per_key * kpw; i += THREADS) {
                const int k = i / per_key;            /* key within the group   */
                const int e = i - k * per_key;        /* (bank, level, bit)     */
                const int bank = e / (g_depth * 2);
                const int lb = e - bank * (g_depth * 2);   /* 2*level + bit       */
                int key = g_key_first + k;
                if (key > g_key_last) key = g_key_last;
                const int level = lb >> 1, bit = lb & 1;
                const uint32_t slot = p.key_compact ? 2u + 4u * (uint32_t)level + 2u * (uint32_t)bank + (uint32_t)bit
                                                    : (bank ? 65u : 1u) + (uint32_t)lb;
                const uint4 v = __ldg(p.keys + (size_t)key * p.key_stride_v + slot);
                cw_s[((level * 2 + bank) * 2 + bit) * 32 + k] = v;
                if (level == 0) cwlo_s[(bank * 2 + bit) * 32 + k] = v.x;
            }
            if (tid < kpw) {
                int key = g_key_first + tid;
                if (key > g_key_last) key = g_key_last;
                root_s[tid] = __ldg(p.keys + (size_t)key * p.key_stride_v + p.key_root_v);
            }
        }
        __syncthreads();
        if (!has_work) continue;

        const int key = g_key_first + kslot;
        env.key_valid = key <= g_key_last;
        if (MODE == MODE_FUSED || MODE == MODE_FUSED_TMA || GROUPED) {
#pragma unroll
            for (int e = 0; e < 4 * NV; e++) env.acc[e] = 0;
        } else if (MODE == MODE_EXPAND) {
            env.share_row = p.shares + (size_t)(env.key_valid ? key : 0) * p.n;
        }
        const uint4 rv = root_s[kslot];
        const Seed root = make_seed(rv.x, rv.y, rv.z, rv.w);

        /* SMALL items (<= 15 node pairs) draw their tickets one draw ahead, so the atomic's round trip
         * to L2 overlaps the items being expanded instead of stalling the warp between items.  Big items
         * draw when they are done: holding a ticket for the length of a 127-pair item makes the hand-out
         * one item less adaptive at the end of a key group (measured: +0.6 % kernel time at n = 2^20,
         * profiles/r2_kernel_regression_bisect.txt), and the atomic's latency is nothing against it.
         * A draw takes a CHUNK of consecutive items, sized from what is left: (remaining / 8x the
         * warps of the grid), between 1 and 8 -- guided self-scheduling: big early chunks when a key
         * group holds many more items than the grid has warps, single items at the end keep the tail
         * fine-grained.  (Cutting a group's tickets into several counters was tried for the case of
         * one or two key groups per GPU and measured slower: profiles/r2_ticket_split_ab.txt.) */
        const uint32_t grid_warps = gridDim.x * (uint32_t)(THREADS / 32);
        const bool chunked = quota == 0xffffffffu;          /* the balanced top round counts single tickets */
        const bool ahead = g_s <= 4;
        uint32_t chunk = 1;
        if (chunked) chunk = min(8u, max(1u, g_tickets / (8u * grid_warps)));
        uint32_t t_raw = 0;
        bool draw = taken < quota;
        if (draw && lane == 0) t_raw = atomicAdd(ph.counters + kg, chunk);
        while (draw) {
            const uint32_t t0 = __shfl_sync(0xffffffffu, t_raw, 0);
            if (t0 >= g_tickets) break;
            const uint32_t t1 = min(t0 + chunk, g_tickets);
            taken += t1 - t0;
            draw = taken < quota;
            if (chunked) chunk = min(8u, max(1u, (g_tickets - t1) / (8u * grid_warps)));
            if (ahead && draw && lane == 0) t_raw = atomicAdd(ph.counters + kg, chunk);
          for (uint32_t t = t0; t < t1; t++) {
            const uint32_t q = (t << spw_log2) + sslot;   /* this lane's subtree */
            Seed start = root;
            if (ph.frontier_in != nullptr) {
                /* written earlier in this launch (before the grid barrier) or by the previous one:
                 * read through L2, never a stale L1 line */
                const uint4 fv = __ldcg(ph.frontier_in + ((size_t)kg * p.nfront + (q >> ph.front_shift)) * kpw + kslot);
                start = make_seed(fv.x, fv.y, fv.z, fv.w);
            }
            const Seed r = walk_down<PRF>(env, start, g_walk_first, g_walk_steps, ph.sub_first + q);
            if (MODE == MODE_FRONTIER) {
                env.front_out = p.frontier_out + ((size_t)kg * p.nfront + ((size_t)q << g_s)) * kpw + kslot;
                eval_subtree<PRF, true>(env, r, g_s, ph.level_base);
            } else {
                env.rows = g_table + ((size_t)q << g_s) * p.row_stride_v + p.col_off_v;
                if constexpr (MODE == MODE_FUSED_TMA) {
                    /* the item's rows are one contiguous run (64-byte rows, breadth-first leaf order) */
                    __syncwarp();                                   /* every lane is done with the previous tile */
                    if (lane == 0) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        const uint32_t bytes = 64u << g_s;
                        tma::mbar_expect_tx(env.tile_bar, bytes);
                        tma::bulk_g2s((uint32_t)__cvta_generic_to_shared(const_cast<uint4 *>(env.tile)), env.rows, bytes, env.tile_bar);
                    }
                    env.tile_pending = true;
                }
                env.pos_base = (ph.sub_first + q) << g_s;
                env.leaf_out = (!GROUPED && p.leaf_cache) ? p.leaf_cache + ((size_t)kg * p.n_local + ((size_t)q << g_s)) * 32 + lane
                                                          : nullptr;
                eval_subtree<PRF, false>(env, r, g_s, 0);
            }
          }
            if (!ahead && draw && lane == 0) t_raw = atomicAdd(ph.counters + kg, chunk);
        }

        if (MODE == MODE_FUSED || MODE == MODE_FUSED_TMA || GROUPED) {
            /* lanes that hold the same key (different subtree slots) fold their partial sums
             * first, so every key receives one red.add per warp and column, not 32/kpw */
            for (int off = kpw; off < 32; off <<= 1) {
#pragma unroll
                for (int e = 0; e < 4 * NV; e++) env.acc[e] += __shfl_xor_sync(0xffffffffu, env.acc[e], off);
            }
            if (QUAD && sslot == 0) {
                /* 4 keys x this lane's column slice; a lane past the group's last key computed that
                 * key's leaves again (clamped correction words), so every key has its own mask */
#pragma unroll
                for (int m = 0; m < 4; m++) {
                    const int key_m = g_key_first + (kslot ^ m);
                    if (key_m > g_key_last) continue;
                    uint32_t *o = p.out + (size_t)key_m * p.out_stride + p.col_off;
#pragma unroll
                    for (int c = 0; c < NV / 4; c++)
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            const uint32_t col = 4u * (4u * c + env.qlane) + e;
                            if (col < p.ncols) atomicAdd(o + col, env.acc[16 * c + 4 * m + e]);
                        }
                }
            } else if (!QUAD && env.key_valid && sslot == 0) {
                uint32_t *o = p.out + (size_t)key * p.out_stride + p.col_off;
#pragma unroll
                for (int e = 0; e < 4 * NV; e++)
                    if ((uint32_t)e < p.ncols) atomicAdd(o + e, env.acc[e]);
            }
        }
        __syncthreads();   /* everyone done with this group's correction words */
    }
}

template <int PRF, int NV, int MODE>
__global__ void __launch_bounds__((KernelShape<PRF, NV>::THREADS), (KernelShape<PRF, NV>::MIN_BLOCKS))
dpf_eval_kernel(const __grid_constant__ EvalParams p)
{
    constexpr int THREADS = KernelShape<PRF, NV>::THREADS;
    const int tid = threadIdx.x;
    unsigned long long *stamp = (p.timing != nullptr && tid == 0) ? p.timing + (size_t)blockIdx.x * 8 : nullptr;
    if (stamp) stamp[0] = global_ns();

    typename TablePolicy<PRF>::type ta;
    if constexpr (PRF == PRF_AES128) {
        /* replicate Te0..Te3 across the 32 banks: entry v, lane L */
        const uint32_t tab = (uint32_t)__cvta_generic_to_shared(g_dyn_smem + p.off_tab);
        if ((tab & 0xffffu) != 0) __trap();   /* layout contract with the host planner */
        for (int i = tid; i < 256 * 32; i += THREADS) {
            const uint32_t v = c_te0[i >> 5];
            unsigned char *e = g_dyn_smem + p.off_tab + (i >> 5) * 256 + (i & 31) * 4;
            *reinterpret_cast<uint32_t *>(e) = v;
            *reinterpret_cast<uint32_t *>(e + 128) = __funnelshift_l(v, v, 8);
            *reinterpret_cast<uint32_t *>(e + 65536) = __funnelshift_l(v, v, 16);
            *reinterpret_cast<uint32_t *>(e + 65536 + 128) = __funnelshift_l(v, v, 24);
        }
        ta.lanebase = tab + (tid & 31) * 4;
    }

    if constexpr (MODE != MODE_FRONTIER) {
        if (p.fuse_top) {
            /* single-launch pipeline: clear this launch's accumulators and main-phase tickets,
             * expand the top of every key's tree into the frontier, meet at the grid barrier */
            const uint64_t gtid = (uint64_t)blockIdx.x * THREADS + tid, gthreads = (uint64_t)gridDim.x * THREADS;
            for (uint64_t i = gtid; i < p.zero_a_words; i += gthreads) p.zero_a[i] = 0u;
            for (uint64_t i = gtid; i < p.zero_b_words; i += gthreads) p.zero_b[i] = 0u;
            if (stamp) stamp[1] = global_ns();
            if (p.top.nsub != 0) {
                /* round 1: every block takes its even share (warp w: quota/nwarps, +1 for the first
                 * quota%nwarps warps); round 2: whatever is left, first come first served */
                constexpr uint32_t NW = THREADS / 32;
                const uint32_t w = (uint32_t)tid >> 5;
                uint32_t bq = p.top_block_quota;
                const uint32_t kgs = (uint32_t)p.key_groups;
                if (bq != 0x7fffffffu && gridDim.x >= kgs) {
                    /* blocks start at key group blockIdx % key_groups: the nb blocks that start at a
                     * group share its tickets exactly, so round 1 leaves nothing behind */
                    const uint32_t nb = gridDim.x / kgs + ((blockIdx.x % kgs) < (gridDim.x % kgs) ? 1u : 0u);
                    const uint32_t tickets = p.top.nsub >> (5 - p.kpw_log2);
                    bq = (tickets + nb - 1) / nb;
                }
                run_phase<PRF, 4, THREADS, MODE_FRONTIER>(p, p.top, ta, bq / NW + (w < bq % NW ? 1u : 0u));
                run_phase<PRF, 4, THREADS, MODE_FRONTIER>(p, p.top, ta);
            }
            if (stamp) stamp[2] = global_ns();
            grid_barrier(p.grid_bar, p.grid_bar_target);
            if (stamp) stamp[3] = global_ns();
            if (blockIdx.x == 0)   /* nobody draws top-phase tickets any more: re-arm them for the next launch */
                for (uint32_t i = tid; i < p.rearm_words; i += THREADS) p.rearm[i] = 0u;
        }
    }
    /* ChaCha measured 0.5-1.2 % slower with the quad MAC layout on a B200 (n = 2^16 and 2^20,
     * B = 512; AES +3.5 %, Salsa +0.4 %), so it keeps the per-lane layout */
    constexpr bool QUAD_MAC = PRF != PRF_CHACHA20;
    if constexpr (QUAD_MAC && (MODE == MODE_FUSED || MODE == MODE_GROUPED || MODE == MODE_FUSED_TMA)) {
        /* kpw_log2 is the same for the whole launch: one of the two MAC layouts runs */
        if (p.kpw_log2 >= 2) run_phase<PRF, NV, THREADS, MODE, true>(p, p.main, ta);
        else run_phase<PRF, NV, THREADS, MODE, false>(p, p.main, ta);
    } else {
        run_phase<PRF, NV, THREADS, MODE>(p, p.main, ta);
    }
    if (stamp) stamp[4] = global_ns();
}

/* MAC-only pass for wide entries: leaves come from the cache written by the first fused
 * pass, rows are broadcast loads as in the fused kernel.  One warp = 32 keys x one range
 * of leaf positions; pure streaming (HBM/L2 -> IMAD), no PRF work. */
template <int NV>
__global__ void __launch_bounds__(256, 2) dpf_mac_kernel(const __grid_constant__ MacParams p)
{
    const int lane = threadIdx.x & 31;
    const uint64_t warp_global = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t warps_total = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t items = (uint64_t)p.key_groups * p.ranges_per_group;
    const uint64_t len = (p.n_local + p.ranges_per_group - 1) / p.ranges_per_group;
    for (uint64_t w = warp_global; w < items; w += warps_total) {
        /* range is the fast index (key-group-fast ordering measured slower: 30.4 vs 29.2 ms at E=128) */
        const uint32_t kg = (uint32_t)(w / p.ranges_per_group);
        const uint32_t r = (uint32_t)(w - (uint64_t)kg * p.ranges_per_group);
        const uint64_t begin = (uint64_t)r * len;
        const uint64_t end = begin + len < p.n_local ? begin + len : p.n_local;
        uint32_t acc[4 * NV];
#pragma unroll
        for (int e = 0; e < 4 * NV; e++) acc[e] = 0;
        const uint32_t *leaf = p.leaf_cache + ((size_t)kg * p.n_local + begin) * 32 + lane;
        const uint4 *row = p.table + begin * p.row_stride_v + p.col_off_v;
        uint64_t pos = begin;
        for (; pos + 4 <= end; pos += 4) {   /* 4 leaves per trip: 4 independent load streams in flight */
            uint32_t v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) v[u] = __ldg(leaf + 32 * u);
#pragma unroll
            for (int j = 0; j < NV; j++) {
                uint4 t[4];
#pragma unroll
                for (int u = 0; u < 4; u++) t[u] = __ldg(row + (size_t)u * p.row_stride_v + j);
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    acc[4 * j + 0] += v[u] * t[u].x;
                    acc[4 * j + 1] += v[u] * t[u].y;
                    acc[4 * j + 2] += v[u] * t[u].z;
                    acc[4 * j + 3] += v[u] * t[u].w;
                }
            }
            leaf += 128;
            row += (size_t)4 * p.row_stride_v;
        }
        for (; pos < end; pos++) {
            const uint32_t v = __ldg(leaf);
#pragma unroll
            for (int j = 0; j < NV; j++) {
                const uint4 t = __ldg(row + j);
                acc[4 * j + 0] += v * t.x;
                acc[4 * j + 1] += v * t.y;
                acc[4 * j + 2] += v * t.z;
                acc[4 * j + 3] += v * t.w;
            }
            leaf += 32;
            row += p.row_stride_v;
        }
        const int key = (int)kg * 32 + lane;
        if (key < p.nkeys) {
            uint32_t *o = p.out + (size_t)key * p.out_stride + p.col_off;
#pragma unroll
            for (int e = 0; e < 4 * NV; e++)
                if ((uint32_t)e >= p.col_skip && (uint32_t)e < p.ncols) atomicAdd(o + e, acc[e]);
        }
    }
}

/* ---- TMA-staged MAC pass ---------------------------------------------------------------------
 * Same arithmetic as dpf_mac_kernel, organised as a producer/consumer pipeline: one warp issues
 * cp.async.bulk copies (table-row slices and cached leaves, global -> shared, completion counted
 * on an mbarrier), eight consumer warps -- one key group each, all on the SAME leaf positions,
 * so a row slice staged once is multiplied against 8 x 32 keys -- do LDS + IMAD only.  The
 * register-staged variant above is latency bound (16 dependent load phases per trip); this one
 * is bound by the FMA pipe. */

template <int NV>
struct MacTmaShape {
    enum { P = 32, STAGES = 3, GROUPS = 8, ROW_BYTES = NV * 16, LEAF_TILE = P * 128,
           STAGE_BYTES = GROUPS * LEAF_TILE + P * ROW_BYTES, SMEM = STAGES * STAGE_BYTES + 64,
           THREADS = (GROUPS + 1) * 32 };
};

template <int NV>
__global__ void __launch_bounds__(MacTmaShape<NV>::THREADS, 1) dpf_mac_tma_kernel(const __grid_constant__ MacParams p)
{
    typedef MacTmaShape<NV> S;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(g_dyn_smem);
    const uint32_t bars = smem0 + S::STAGES * S::STAGE_BYTES;   /* full[STAGES], empty[STAGES] */
    if (threadIdx.x == 0) {
        for (int i = 0; i < S::STAGES; i++) {
            tma::mbar_init(bars + 8 * i, 1);                       /* producer's expect_tx arrival */
            tma::mbar_init(bars + 8 * (S::STAGES + i), S::GROUPS); /* one arrival per consumer warp */
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const uint32_t kg_blocks = ((uint32_t)p.key_groups + S::GROUPS - 1) / S::GROUPS;
    const uint64_t items = (uint64_t)kg_blocks * p.ranges_per_group;
    const uint64_t len = (p.n_local + p.ranges_per_group - 1) / p.ranges_per_group;
    uint32_t seq = 0;   /* tiles issued / consumed so far: stage = seq % STAGES, phase = (seq / STAGES) & 1 */

    for (uint64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const uint32_t kgb = (uint32_t)(it / p.ranges_per_group);
        const uint32_t r = (uint32_t)(it - (uint64_t)kgb * p.ranges_per_group);
        const uint64_t begin = (uint64_t)r * len;
        const uint64_t end = begin + len < p.n_local ? begin + len : p.n_local;
        const uint32_t kg0 = kgb * S::GROUPS;
        const uint32_t ngroups = min((uint32_t)S::GROUPS, (uint32_t)p.key_groups - kg0);

        if (warp == S::GROUPS) {
            /* ===== producer warp ===== */
            for (uint64_t pos = begin; pos < end; pos += S::P, seq++) {
                const uint32_t stage = seq % S::STAGES, phase = (seq / S::STAGES) & 1u;
                const uint32_t cnt = (uint32_t)min((uint64_t)S::P, end - pos);
                const uint32_t sbase = smem0 + stage * S::STAGE_BYTES;
                const uint32_t full = bars + 8 * stage, empty = bars + 8 * (S::STAGES + stage);
                tma::mbar_wait(empty, phase ^ 1u);     /* consumers have released this stage */
                if (lane == 0) tma::mbar_expect_tx(full, cnt * (128u * ngroups + S::ROW_BYTES));
                __syncwarp();
                if ((uint32_t)lane < ngroups)          /* cached leaves: one contiguous slab per key group */
                    tma::bulk_g2s(sbase + lane * S::LEAF_TILE,
                                  p.leaf_cache + ((size_t)(kg0 + lane) * p.n_local + pos) * 32, cnt * 128u, full);
                for (uint32_t i = lane; i < cnt; i += 32)   /* one row slice per leaf position */
                    tma::bulk_g2s(sbase + S::GROUPS * S::LEAF_TILE + i * S::ROW_BYTES,
                                  p.table + (pos + i) * p.row_stride_v + p.col_off_v, S::ROW_BYTES, full);
            }
        } else {
            /* ===== consumer warps: warp w = key group kg0 + w ===== */
            const bool active = (uint32_t)warp < ngroups;
            uint32_t acc[4 * NV];
#pragma unroll
            for (int e = 0; e < 4 * NV; e++) acc[e] = 0;
            for (uint64_t pos = begin; pos < end; pos += S::P, seq++) {
                const uint32_t stage = seq % S::STAGES, phase = (seq / S::STAGES) & 1u;
                const uint32_t cnt = (uint32_t)min((uint64_t)S::P, end - pos);
                const unsigned char *sbase = g_dyn_smem + stage * S::STAGE_BYTES;
                tma::mbar_wait(bars + 8 * stage, phase);   /* the bytes have landed */
                if (active) {
                    const uint32_t *leaf = reinterpret_cast<const uint32_t *>(sbase + warp * S::LEAF_TILE) + lane;
                    const uint4 *rows = reinterpret_cast<const uint4 *>(sbase + S::GROUPS * S::LEAF_TILE);
#pragma unroll 2
                    for (uint32_t i = 0; i < cnt; i++) {
                        const uint32_t v = leaf[i * 32];
#pragma unroll
                        for (int j = 0; j < NV; j++) {
                            const uint4 t = rows[i * NV + j];
                            acc[4 * j + 0] += v * t.x;
                            acc[4 * j + 1] += v * t.y;
                            acc[4 * j + 2] += v * t.z;
                            acc[4 * j + 3] += v * t.w;
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) tma::mbar_arrive(bars + 8 * (S::STAGES + stage));
            }
            const int key = (int)(kg0 + warp) * 32 + lane;
            if (active && key < p.nkeys) {
                uint32_t *o = p.out + (size_t)key * p.out_stride + p.col_off;
#pragma unroll
                for (int e = 0; e < 4 * NV; e++)
                    if ((uint32_t)e >= p.col_skip && (uint32_t)e < p.ncols) atomicAdd(o + e, acc[e]);
            }
        }
    }
}

__global__ void __launch_bounds__(256) sum_partials_kernel(uint32_t *__restrict__ dst, const PeerParts parts, size_t words)
{
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (size_t)gridDim.x * blockDim.x;
    if ((words & 3u) == 0) {   /* results are [B][E] int32 from cudaMalloc: 16-byte aligned whenever the count allows */
        uint4 *d4 = reinterpret_cast<uint4 *>(dst);
        for (size_t i = tid; i < words / 4; i += nthr) {
            uint4 a = d4[i];
            for (int k = 0; k < parts.n; k++) {
                const uint4 b = __ldcg(reinterpret_cast<const uint4 *>(parts.p[k]) + i);   /* peer memory over NVLink */
                a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
            }
            d4[i] = a;
        }
    } else {
        for (size_t i = tid; i < words; i += nthr) {
            uint32_t a = dst[i];
            for (int k = 0; k < parts.n; k++) a += __ldcg(parts.p[k] + i);
            dst[i] = a;
        }
    }
}

__global__ void probe_smem_kernel(uint32_t *out)
{
    if (threadIdx.x == 0) *out = (uint32_t)__cvta_generic_to_shared(g_dyn_smem);
}

__global__ void permute_table_kernel(const int32_t *__restrict__ stage, int32_t *__restrict__ table,
                                     uint64_t rows, int bits, int cols, int stride)
{
    const uint64_t total = rows * (uint64_t)cols;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t q = i / (uint64_t)cols;
        const int c = (int)(i - q * (uint64_t)cols);
        const uint64_t src = bits ? (uint64_t)(__brev((uint32_t)q) >> (32 - bits)) : 0;
        table[q * (uint64_t)stride + c] = stage[src * (uint64_t)cols + c];
    }
}

template <int PRF, int NV, int MODE>
cudaError_t launch_one(const EvalParams &p, int grid, size_t smem, cudaStream_t stream)
{
    auto kern = dpf_eval_kernel<PRF, NV, MODE>;
    /* function attributes are per device and sticky: set them once per (device, size); contexts
     * on different host threads may race here, hence the atomics (a duplicate set is harmless) */
    static std::atomic<int> configured[64];   /* smem bytes + 1 last configured on each device, 0 = never */
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || configured[dev].load(std::memory_order_acquire) != (int)smem + 1) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        /* the kernels live in shared memory; L1 only sees broadcast table rows */
        e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev].store((int)smem + 1, std::memory_order_release);
    }
    if (p.fuse_top) {
        void *args[] = {const_cast<EvalParams *>(&p)};
        return cudaLaunchCooperativeKernel(reinterpret_cast<const void *>(kern), dim3((unsigned)grid),
                                           dim3((unsigned)(KernelShape<PRF, NV>::THREADS)), args, smem, stream);
    }
    kern<<<grid, (KernelShape<PRF, NV>::THREADS), smem, stream>>>(p);
    return cudaGetLastError();
}

template <int PRF, int NV, int MODE>
cudaError_t max_smem_one(int *bytes)
{
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, dpf_eval_kernel<PRF, NV, MODE>);
    if (e != cudaSuccess) return e;
    int dev = 0, optin = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
    *bytes = optin - (int)a.sharedSizeBytes;
    return cudaSuccess;
}

/* (prf, nv, mode) -> instantiation; modes 1 and 2 never touch the table, so NV = 4 only; grouped
 * evaluation takes 16 columns per pass */
template <int PRF>
cudaError_t launch_prf(int nv, int mode, const EvalParams &p, int grid, size_t smem, cudaStream_t stream)
{
    if (mode == MODE_EXPAND) return launch_one<PRF, 4, MODE_EXPAND>(p, grid, smem, stream);
    if (mode == MODE_FRONTIER) return launch_one<PRF, 4, MODE_FRONTIER>(p, grid, smem, stream);
    if (mode == MODE_GROUPED) return launch_one<PRF, 4, MODE_GROUPED>(p, grid, smem, stream);
    if (mode == MODE_FUSED_TMA) {
        if constexpr (PRF == PRF_AES128) return cudaErrorInvalidValue;    /* no shared memory left beside the tables */
        else return launch_one<PRF, 4, MODE_FUSED_TMA>(p, grid, smem, stream);
    }
    if (nv == 4) return launch_one<PRF, 4, MODE_FUSED>(p, grid, smem, stream);
    if (nv == 8) return launch_one<PRF, 8, MODE_FUSED>(p, grid, smem, stream);
    if (nv == 16) return launch_one<PRF, 16, MODE_FUSED>(p, grid, smem, stream);
    return cudaErrorInvalidValue;
}

template <int PRF>
cudaError_t max_smem_prf(int nv, int mode, int *bytes)
{
    if (mode == MODE_EXPAND) return max_smem_one<PRF, 4, MODE_EXPAND>(bytes);
    if (mode == MODE_FRONTIER) return max_smem_one<PRF, 4, MODE_FRONTIER>(bytes);
    if (mode == MODE_GROUPED) return max_smem_one<PRF, 4, MODE_GROUPED>(bytes);
    if (mode == MODE_FUSED_TMA) {
        if constexpr (PRF == PRF_AES128) return cudaErrorInvalidValue;
        else return max_smem_one<PRF, 4, MODE_FUSED_TMA>(bytes);
    }
    if (nv == 4) return max_smem_one<PRF, 4, MODE_FUSED>(bytes);
    if (nv == 8) return max_smem_one<PRF, 8, MODE_FUSED>(bytes);
    if (nv == 16) return max_smem_one<PRF, 16, MODE_FUSED>(bytes);
    return cudaErrorInvalidValue;
}

}  // namespace

int eval_threads(int prf, int nv)
{
    if (prf == PRF_AES128) return nv <= 8 ? DPF_AES_THREADS : 256;
    return nv <= 8 ? 256 : 384;
}

int eval_min_blocks(int prf, int nv)
{
    if (prf == PRF_AES128) return 1;
    return nv <= 8 ? 2 : 1;
}

cudaError_t probe_dynamic_smem_base(uint32_t *base, cudaStream_t stream)
{
    uint32_t *d = nullptr;
    cudaError_t e = cudaMalloc(&d, sizeof(uint32_t));
    if (e != cudaSuccess) return e;
    probe_smem_kernel<<<1, 32, 16, stream>>>(d);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(base, d, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    cudaFree(d);
    return e;
}

cudaError_t upload_aes_table(const uint32_t *te0_256)
{
    return cudaMemcpyToSymbol(c_te0, te0_256, 256 * sizeof(uint32_t));
}

cudaError_t launch_eval(int prf, int nv, int mode, const EvalParams &p, int grid, size_t smem, cudaStream_t stream)
{
    switch (prf) {
    case PRF_DUMMY: return launch_prf<PRF_DUMMY>(nv, mode, p, grid, smem, stream);
    case PRF_SALSA20: return launch_prf<PRF_SALSA20>(nv, mode, p, grid, smem, stream);
    case PRF_CHACHA20: return launch_prf<PRF_CHACHA20>(nv, mode, p, grid, smem, stream);
    case PRF_AES128: return launch_prf<PRF_AES128>(nv, mode, p, grid, smem, stream);
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t eval_max_smem(int prf, int nv, int mode, int *bytes)
{
    switch (prf) {
    case PRF_DUMMY: return max_smem_prf<PRF_DUMMY>(nv, mode, bytes);
    case PRF_SALSA20: return max_smem_prf<PRF_SALSA20>(nv, mode, bytes);
    case PRF_CHACHA20: return max_smem_prf<PRF_CHACHA20>(nv, mode, bytes);
    case PRF_AES128: return max_smem_prf<PRF_AES128>(nv, mode, bytes);
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_mac_tma(const MacParams &p, int grid, cudaStream_t stream)
{
    typedef MacTmaShape<16> S;
    auto kern = dpf_mac_tma_kernel<16>;
    static std::atomic<int> configured[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || !configured[dev].load(std::memory_order_acquire)) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::SMEM);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev].store(1, std::memory_order_release);
    }
    kern<<<grid, (int)S::THREADS, (int)S::SMEM, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_mac(int nv, const MacParams &p, int grid, cudaStream_t stream)
{
    if (nv == 4) dpf_mac_kernel<4><<<grid, 256, 0, stream>>>(p);
    else if (nv == 8) dpf_mac_kernel<8><<<grid, 256, 0, stream>>>(p);
    else if (nv == 16) dpf_mac_kernel<16><<<grid, 256, 0, stream>>>(p);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

cudaError_t launch_sum_partials(uint32_t *dst, const PeerParts &parts, size_t words, cudaStream_t stream)
{
    if (parts.n <= 0 || words == 0) return cudaSuccess;
    int grid = (int)std::min<size_t>((words / 4 + 255) / 256 + 1, 148 * 4);
    sum_partials_kernel<<<grid, 256, 0, stream>>>(dst, parts, words);
    return cudaGetLastError();
}

cudaError_t launch_permute_table(const int32_t *stage, int32_t *table, uint64_t rows, int bits,
                                 int cols, int stride, cudaStream_t stream)
{
    const uint64_t total = rows * (uint64_t)cols;
    int grid = (int)((total + 255) / 256);
    if (grid > 148 * 16) grid = 148 * 16;
    if (grid < 1) grid = 1;
    permute_table_kernel<<<grid, 256, 0, stream>>>(stage, table, rows, bits, cols, stride);
    return cudaGetLastError();
}

}  // namespace b200dpf
