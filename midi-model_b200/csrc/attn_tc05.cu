// Causal attention for the event-level stack on the 5th-gen tensor cores (head_dim 64), forward and backward:
// every matmul is tcgen05.mma with accumulators in TMEM, Q / K / V / dO tiles are staged by TMA (cp.async.bulk.tensor.3d,
// 128B swizzle, zero fill outside the sequence) straight from the packed [rows, 3*hidden] QKV activation, and the
// fp32 softmax math runs on dedicated warps that exchange tiles with the MMA-issuing thread(s) through mbarriers.
// Kernels, in file order:
//   attn_fwd_tc05_kernel         forward: persistent, two query tiles per CTA, thread = row, O in TMEM with a lazy rescale,
//                                ping-pong between the two softmax groups (0.147-0.155 ms per layer at B=8, S=2048)
//   attn_bwd_tc05_kernel         backward: dK, dV and dQ (through a TMA reduce-add), half-tile pipeline
//   attn_bwd_dq_finalize_kernel  fp32 dQ -> bf16
// DESIGN.md 3.1b has the measurements behind these choices and the variants they ruled out.
// Semantics = hf sdpa_attention.py:92-101 (causal, scale d^-1/2): online softmax in fp32, P rounded to bf16
// before P.V, output rounded to bf16, LSE saved for the backward pass.
#include "tc05.cuh"

namespace {
using namespace tc05;

constexpr int D = 64;
constexpr int BQ = 128;    // query rows per tile
constexpr int BK = 128;    // keys per tile
constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

// advance a shared-memory matrix descriptor by `bytes` (start-address field, 16-byte units); smem addresses are
// < 256 KB so the 14-bit field never overflows
__device__ __forceinline__ uint64_t desc_adv(uint64_t d, uint32_t bytes) { return d + (uint64_t)(bytes >> 4); }

struct FwdParams {
    bf16* o;
    float* lse;
    long long o_b, o_r;          // element strides of the output: batch, row (heads are contiguous blocks of 64)
    int batch;
    int n_heads, Sq, Sk, H;      // H = columns between the q, k and v thirds when packed (used for TMA column coords)
    int q_col0, k_col0, v_col0;  // first column of head 0 in each tensor map
    float scale;
    long long* dbg;              // forward phase profile (NULL = off)
};

// ---------------------------------------------------------------------------------------------
// forward: persistent, two query tiles per CTA, thread = one query row.
//   * grid = one CTA per SM; every CTA walks a static, length-balanced list of work items (snake order over the items sorted
//     longest first).  An item = two adjacent 128-row query tiles of one (batch, head); both tiles consume the same K/V
//     stream, so every K/V tile is staged once for 256 query rows.
//   * two softmax groups of 4 warps (one per query tile); a thread owns a whole row of the 128-key score tile, so the row
//     maximum and the row sum never leave its registers (no shared-memory exchange, no named barriers).  The two groups
//     sit pairwise on the four SM sub-partitions and drift out of phase, so one group's MUFU burst overlaps the other's
//     max / convert / store work.
//   * the output accumulates in TMEM (P.V with the accumulate flag); it is rescaled in place only when a row's maximum has
//     grown by more than 2^8 since the reference maximum was taken (lazy rescale: with a stale maximum the probabilities
//     are at most 256, exact in fp32 and harmless in bf16), which in practice happens on the first tiles of a row only.
//   * one MMA-issuing warp per group: S_{j+1} = Q.K^T is issued as soon as the group has read S_j out of TMEM, P.V_j when
//     P_j is in shared memory.  K/V stages are released when both groups' MMAs on them have retired.
//   * ping-pong: the two softmax warps that share an SM sub-partition (same row quarter, different group) take turns in the
//     MUFU-bound half of a tile (pass 2) through a pair of 64-thread named barriers, so that one warp's exponentials run
//     against the other's tile-load / row-maximum / barrier work instead of against its exponentials.
//   warp 0: TMA producer   warps 1, 2: MMA issuers of group 0 / 1   warp 3: TMEM allocator   warps 4..7 / 8..11: softmax
// ---------------------------------------------------------------------------------------------
constexpr int FWD_THREADS = 384;
constexpr int FWD_KVS = 4;                               // K/V stages
constexpr int SF_Q = 0;                                  // 2 x 16 KB
constexpr int SF_P = 32768;                              // 2 x 32 KB (one P tile per group)
constexpr int SF_KV = SF_P + 2 * 32768;                  // FWD_KVS x (K 16 KB + V 16 KB)
constexpr int SF_BAR = SF_KV + FWD_KVS * 32768;
constexpr int SMEM_FWD_BYTES = SF_BAR + 256;
constexpr float RESCALE_LOG2 = 8.f;

struct FwdItem {
    int b, h;
    int q0[2], n[2], nt;      // first query row and number of K/V tiles of each group (0 = group idle), max of the two
};

__device__ __forceinline__ bool fwd_item(const FwdParams& p, int round, FwdItem& it) {
    const int n_qt = (p.Sq + BQ - 1) / BQ, n_pairs = (n_qt + 1) >> 1;
    const int n_bh = p.batch * p.n_heads;
    const int G = gridDim.x, c = blockIdx.x;
    const long long idx = (long long)round * G + ((round & 1) ? G - 1 - c : c);
    if (idx >= (long long)n_pairs * n_bh) return false;
    const int pt = n_pairs - 1 - (int)(idx / n_bh);           // long (late) tile pairs first
    const int bh = (int)(idx % n_bh);
    it.b = bh / p.n_heads; it.h = bh % p.n_heads;
    const int off = p.Sk - p.Sq;
    it.nt = 0;
#pragma unroll
    for (int g = 0; g < 2; g++) {
        const int qt = 2 * pt + g;
        it.q0[g] = qt * BQ;
        int n = 0;
        if (qt < n_qt) {
            n = min((p.Sk + BK - 1) / BK, (it.q0[g] + BQ - 1 + off) / BK + 1);
            if (n < 1) n = 1;
        }
        it.n[g] = n;
        it.nt = max(it.nt, n);
    }
    return true;
}

// PROF: per-phase clock64 sums of the softmax warps into p.dbg (tools/attn_fwd_profile.py through b200_attn_debug_trace)
template <bool PROF>
__global__ void __launch_bounds__(FWD_THREADS, 1)
attn_fwd_tc05_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                     const __grid_constant__ CUtensorMap tmV, const FwdParams p) {
    B200_PDL_TRIGGER();
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SF_BAR);
    uint64_t* kv_full = bars + 0;      // [FWD_KVS]
    uint64_t* kv_empty = bars + 4;     // [FWD_KVS]  one arrival per MMA warp
    uint64_t* q_full = bars + 8;       // [2]
    uint64_t* q_empty = bars + 10;     // [2]
    uint64_t* s_full = bars + 12;      // [2]
    uint64_t* s_empty = bars + 14;     // [2]  4 softmax warps
    uint64_t* p_full = bars + 16;      // [2]  4 softmax warps
    uint64_t* pv_done = bars + 18;     // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 20);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_rounds = (int)(((long long)((p.Sq + BQ - 1) / BQ + 1) / 2 * p.batch * p.n_heads + gridDim.x - 1) / gridDim.x);

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmQ); prefetch_tmap(&tmK); prefetch_tmap(&tmV);
        for (int s = 0; s < FWD_KVS; s++) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 2); }
        for (int g = 0; g < 2; g++) {
            mbar_init(&q_full[g], 1); mbar_init(&q_empty[g], 1); mbar_init(&s_full[g], 1); mbar_init(&s_empty[g], 4);
            mbar_init(&p_full[g], 4); mbar_init(&pv_done[g], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 3) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t T = 0, cq[2] = {0, 0};
            FwdItem it;
            for (int r = 0; r < n_rounds; r++) {
                if (!fwd_item(p, r, it)) continue;
#pragma unroll
                for (int g = 0; g < 2; g++) {
                    if (it.n[g] == 0) continue;
                    mbar_wait(&q_empty[g], (cq[g] & 1) ^ 1);
                    mbar_expect_tx(&q_full[g], BQ * D * 2);
                    tma_load_3d(smem + SF_Q + g * 16384, &tmQ, &q_full[g], p.q_col0 + it.h * D, it.q0[g], it.b);
                    cq[g]++;
                }
                for (int j = 0; j < it.nt; j++, T++) {
                    const int st = T % FWD_KVS;
                    mbar_wait(&kv_empty[st], ((T / FWD_KVS) & 1) ^ 1);
                    uint8_t* sK = smem + SF_KV + st * 32768;
                    mbar_expect_tx(&kv_full[st], 2 * BK * D * 2);
                    tma_load_3d(sK, &tmK, &kv_full[st], p.k_col0 + it.h * D, j * BK, it.b);
                    tma_load_3d(sK + 16384, &tmV, &kv_full[st], p.v_col0 + it.h * D, j * BK, it.b);
                }
            }
        }
    } else if (warp == 1 || warp == 2) {
        if (lane == 0) {
            const int g = warp - 1;
            constexpr uint32_t idesc_s = make_idesc(BQ, BK, false, false);    // S[128 x 128] = Q . K^T
            constexpr uint32_t idesc_pv = make_idesc(BQ, D, false, true);     // O[128 x 64] += P . V (V is [keys, d]: MN-major B)
            const uint32_t tS = tmem_base + g * 128, tO = tmem_base + 256 + g * 64;
            const uint64_t dQ0 = make_smem_desc(smem_u32(smem + SF_Q + g * 16384), 16, 1024);
            const uint64_t dP0 = make_smem_desc(smem_u32(smem + SF_P + g * 32768), 16, 1024);
            uint32_t T = 0, tg = 0, cq = 0;
            auto issue_s = [&](uint32_t Tj) {               // S = Q . K_j^T of the K/V tile with running index Tj
                const int st = Tj % FWD_KVS;
                mbar_wait(&kv_full[st], (Tj / FWD_KVS) & 1);
                const uint64_t dK0 = make_smem_desc(smem_u32(smem + SF_KV + st * 32768), 16, 1024);
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < D / 16; k++) umma_f16(tS, desc_adv(dQ0, k * 32), desc_adv(dK0, k * 32), idesc_s, k > 0);
                umma_commit(&s_full[g]);
            };
            FwdItem it;
            for (int r = 0; r < n_rounds; r++) {
                if (!fwd_item(p, r, it)) continue;
                const int n = g ? it.n[1] : it.n[0];
                if (n > 0) { mbar_wait(&q_full[g], cq & 1); cq++; }
                for (int j = 0; j < it.nt; j++, T++) {
                    const int st = T % FWD_KVS;
                    if (j < n) {
                        if (j == 0) {
                            if (tg > 0) mbar_wait(&s_empty[g], (tg - 1) & 1);      // last tile of the previous item read out
                            issue_s(T);
                            if (n == 1) umma_commit(&q_empty[g]);
                        }
                        if (j + 1 < n) {                                           // S_{j+1} first: the group never waits for it
                            mbar_wait(&s_empty[g], tg & 1);
                            issue_s(T + 1);
                            if (j + 2 == n) umma_commit(&q_empty[g]);
                        }
                        mbar_wait(&p_full[g], tg & 1);
                        tc_fence_after();
                        const uint64_t dV0 = make_smem_desc(smem_u32(smem + SF_KV + st * 32768 + 16384), 16384, 1024);
#pragma unroll
                        for (int kk = 0; kk < BK / 16; kk++)
                            umma_f16(tO, desc_adv(dP0, (kk >> 2) * 16384 + (kk & 3) * 32), desc_adv(dV0, kk * 2048), idesc_pv,
                                     (j > 0 || kk > 0) ? 1u : 0u);
                        umma_commit(&pv_done[g]);
                        umma_commit(&kv_empty[st]);
                        tg++;
                    } else {
                        mbar_wait(&kv_full[st], (T / FWD_KVS) & 1);                 // the other group's tile: just pass the stage on
                        mbar_arrive(&kv_empty[st]);
                    }
                }
            }
        }
    } else if (warp >= 4) {
        const int g = (warp - 4) >> 2;
        const int quarter = warp & 3;
        const int row_t = quarter * 32 + lane;            // row inside the tile == TMEM lane
        const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
        const uint32_t tS = tmem_base + g * 128 + lane_addr, tO = tmem_base + 256 + g * 64 + lane_addr;
        const float sl2 = p.scale * LOG2E;
        const int off = p.Sk - p.Sq;
        uint8_t* sP = smem + SF_P + g * 32768;
        uint32_t tg = 0;
        // ping-pong token of this sub-partition: barrier 1 + 2*quarter + g is the one this warp waits on
        const int bar_mine = 1 + 2 * quarter + g, bar_other = 1 + 2 * quarter + (g ^ 1);
        if (g == 1) asm volatile("bar.arrive %0, 64;" ::"r"(bar_other) : "memory");    // group 0 goes first
        long long pf[8] = {0, 0, 0, 0, 0, 0, 0, 0}, pt = 0;      // PROF: cycles per phase (lane 0), tiles
        const long long pstart = PROF ? clock64() : 0;
        auto mark = [&](int k) {
            if (PROF) { const long long t = clock64(); pf[k] += t - pt; pt = t; }
        };
        pt = pstart;
        FwdItem it;
        for (int r = 0; r < n_rounds; r++) {
            if (!fwd_item(p, r, it)) continue;
            const int n = g ? it.n[1] : it.n[0];
            const int q0 = g ? it.q0[1] : it.q0[0], row = q0 + row_t;
            float m_ref = -INFINITY, l_i = 0.f;
            for (int j = 0; j < it.nt; j++) {
                if (j >= n) {            // the other group's extra tile: keep the token moving
                    asm volatile("bar.sync %0, 64;" ::"r"(bar_mine) : "memory");
                    asm volatile("bar.arrive %0, 64;" ::"r"(bar_other) : "memory");
                    continue;
                }
                const int k0 = j * BK;
                const bool need_mask = (k0 + BK - 1 > q0 + off) || (k0 + BK > p.Sk);
                const int lim0 = min(row + off, p.Sk - 1) - k0;     // last visible column of this row in the tile
                mark(6);
                mbar_wait(&s_full[g], tg & 1);
                tc_fence_after();
                mark(0);
                uint32_t rr[2][32];
                // ---- pass 1: row maximum
                float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
                tmem_ld32(tS, rr[0]);
                tmem_ld_wait();
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    if (c < 3) tmem_ld32(tS + (c + 1) * 32, rr[(c + 1) & 1]);
                    if (need_mask) {
                        const int lim = lim0 - c * 32;
#pragma unroll
                        for (int i = 0; i < 32; i++)
                            mx4[i & 3] = fmaxf(mx4[i & 3], (i > lim) ? -INFINITY : __uint_as_float(rr[c & 1][i]));
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; i++) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(rr[c & 1][i]));
                    }
                    if (c < 3) tmem_ld_wait();
                }
                const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
                // ---- reference maximum; P buffer and O are free / stable once P.V of the previous tile has retired
                const bool need = (mx - m_ref) * sl2 > RESCALE_LOG2;       // true on the first tile (m_ref = -inf)
                mark(1);
                if (j > 0) {
                    mbar_wait(&pv_done[g], (tg - 1) & 1);
                    tc_fence_after();
                }
                if (__any_sync(0xffffffffu, need)) {
                    const float m_new = need ? mx : m_ref;
                    if (j > 0) {
                        const float alpha = need ? exp2f((m_ref - m_new) * sl2) : 1.f;
#pragma unroll
                        for (int c = 0; c < 2; c++) {
                            tmem_ld32(tO + c * 32, rr[0]);
                            tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 32; i++) rr[0][i] = __float_as_uint(__uint_as_float(rr[0][i]) * alpha);
                            tmem_st32(tO + c * 32, rr[0]);
                        }
                        tmem_st_wait();
                        l_i *= alpha;
                    }
                    m_ref = m_new;
                }
                const float msc = m_ref * sl2;
                // ---- pass 2: probabilities -> bf16 -> swizzled P tile in shared memory
                mark(2);
                asm volatile("bar.sync %0, 64;" ::"r"(bar_mine) : "memory");
                mark(3);
                float rs4[4] = {0.f, 0.f, 0.f, 0.f};
                tmem_ld32(tS, rr[0]);
                tmem_ld_wait();
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    if (c < 3) tmem_ld32(tS + (c + 1) * 32, rr[(c + 1) & 1]);
                    uint32_t pk[16];
                    if (need_mask) {
                        const int lim = lim0 - c * 32;
#pragma unroll
                        for (int i = 0; i < 32; i += 2) {
                            const float p0 = (i > lim) ? 0.f : ex2_approx(fmaf(__uint_as_float(rr[c & 1][i]), sl2, -msc));
                            const float p1 = (i + 1 > lim) ? 0.f : ex2_approx(fmaf(__uint_as_float(rr[c & 1][i + 1]), sl2, -msc));
                            rs4[(i >> 1) & 3] += p0 + p1;
                            pk[i >> 1] = pack2(p0, p1);
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; i += 2) {
                            const float p0 = ex2_approx(fmaf(__uint_as_float(rr[c & 1][i]), sl2, -msc));
                            const float p1 = ex2_approx(fmaf(__uint_as_float(rr[c & 1][i + 1]), sl2, -msc));
                            rs4[(i >> 1) & 3] += p0 + p1;
                            pk[i >> 1] = pack2(p0, p1);
                        }
                    }
                    // keys c*32 .. +31 of this row: atom (c >> 1), 16-byte chunks (c & 1) * 4 .. + 3
                    uint8_t* rowp = sP + (c >> 1) * 16384 + row_t * 128;
#pragma unroll
                    for (int v = 0; v < 4; v++) {
                        const int chunk = (c & 1) * 4 + v;
                        *reinterpret_cast<uint4*>(rowp + ((chunk ^ (row_t & 7)) << 4)) =
                            make_uint4(pk[4 * v], pk[4 * v + 1], pk[4 * v + 2], pk[4 * v + 3]);
                    }
                    if (c < 3) tmem_ld_wait();
                    if (c == 2) {                      // the whole S tile is in registers: the tensor pipe may overwrite it
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&s_empty[g]);
                    }
                }
                asm volatile("bar.arrive %0, 64;" ::"r"(bar_other) : "memory");
                mark(4);
                l_i += (rs4[0] + rs4[1]) + (rs4[2] + rs4[3]);
                tc_fence_before();
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&p_full[g]);
                tg++;
                mark(5);
            }
            if (n == 0) continue;
            // ---- epilogue of the item: O / l -> bf16
            mbar_wait(&pv_done[g], (tg - 1) & 1);
            tc_fence_after();
            const float inv = l_i > 0.f ? 1.f / l_i : 0.f;
            bf16* dst = p.o + it.b * p.o_b + (long long)row * p.o_r + it.h * D;
#pragma unroll
            for (int c = 0; c < 2; c++) {
                uint32_t r[32];
                tmem_ld32(tO + c * 32, r);
                tmem_ld_wait();
                if (row < p.Sq) {
#pragma unroll
                    for (int v = 0; v < 4; v++) {
                        float f[8];
#pragma unroll
                        for (int i = 0; i < 8; i++) f[i] = __uint_as_float(r[v * 8 + i]) * inv;
                        *reinterpret_cast<uint4*>(dst + c * 32 + v * 8) = pack8(f);
                    }
                }
            }
            if (p.lse && row < p.Sq) p.lse[((long long)it.b * p.n_heads + it.h) * p.Sq + row] = m_ref * p.scale + logf(l_i);
            // the next item's first P.V (accumulate = 0) overwrites O only after this thread's p_full arrival: ordered
            tc_fence_before();
        }
        if (g == 0) asm volatile("bar.sync %0, 64;" ::"r"(bar_mine) : "memory");    // consume the last token
        if (PROF && lane == 0 && p.dbg) {
            mark(6);                                   // [6] = epilogues + item bookkeeping + dummy token passes
            for (int k = 0; k < 7; k++) atomicAdd((unsigned long long*)&p.dbg[g * 16 + k], (unsigned long long)pf[k]);
            atomicAdd((unsigned long long*)&p.dbg[g * 16 + 7], (unsigned long long)(clock64() - pstart));
            atomicAdd((unsigned long long*)&p.dbg[g * 16 + 8], (unsigned long long)tg);
            atomicAdd((unsigned long long*)&p.dbg[g * 16 + 9], 1ull);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 3) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

}   // namespace

static long long* g_attn_dbg = nullptr;

// 3-D bf16 tensor map {cols, rows per sequence, batch} with 128B swizzle: rows outside a sequence are zero-filled
int tc05_make_tmap_3d(CUtensorMap* tm, const void* ptr, uint64_t cols, uint64_t rows, uint64_t batch, uint64_t row_pitch,
                      uint64_t batch_pitch, uint32_t box_cols, uint32_t box_rows);
int tc05_make_tmap_3d_f32(CUtensorMap* tm, const void* ptr, uint64_t cols, uint64_t rows, uint64_t batch, uint64_t row_pitch,
                          uint64_t batch_pitch, uint32_t box_cols, uint32_t box_rows);

// q, k, v: [batch, S, heads*64] views (row pitch / batch pitch in elements) of e.g. the packed QKV activation
extern "C" int b200_attn_causal_fwd_tc(const void* q, const void* k, const void* v, void* o, float* lse,
                                       const long long* strides /* 4 x {b,r,h}: q,k,v,o */, int batch, int n_heads, int Sq,
                                       int Sk, int head_dim, float scale, cudaStream_t stream) {
    B200_CHECK_ARG(head_dim == D, "attn_causal_fwd_tc: head_dim %d unsupported (64 only)", head_dim);
    B200_CHECK_ARG(Sk >= Sq, "attn_causal_fwd_tc: Sk must be >= Sq");
    for (int i = 0; i < 4; i++)
        B200_CHECK_ARG(strides[3 * i + 2] == D, "attn_causal_fwd_tc: heads must be contiguous blocks of 64 columns");
    if (batch == 0 || Sq == 0) return B200_OK;
    const long long W = (long long)n_heads * D;
    CUtensorMap tmQ, tmK, tmV;
    int rc;
    if ((rc = tc05_make_tmap_3d(&tmQ, q, W, Sq, batch, strides[1], strides[0], D, BQ))) return rc;
    if ((rc = tc05_make_tmap_3d(&tmK, k, W, Sk, batch, strides[4], strides[3], D, BK))) return rc;
    if ((rc = tc05_make_tmap_3d(&tmV, v, W, Sk, batch, strides[7], strides[6], D, BK))) return rc;
    FwdParams p;
    p.o = (bf16*)o; p.lse = lse; p.o_b = strides[9]; p.o_r = strides[10];
    p.batch = batch; p.n_heads = n_heads; p.Sq = Sq; p.Sk = Sk; p.H = (int)W;
    p.q_col0 = p.k_col0 = p.v_col0 = 0;
    p.scale = scale;
    p.dbg = g_attn_dbg;
    static bool configured = false;
    if (!configured) {
        B200_CUDA(cudaFuncSetAttribute(attn_fwd_tc05_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_FWD_BYTES),
                  "attn_tc smem");
        B200_CUDA(cudaFuncSetAttribute(attn_fwd_tc05_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_FWD_BYTES),
                  "attn_tc smem");
        configured = true;
    }
    const long long items = (long long)(((Sq + BQ - 1) / BQ + 1) / 2) * batch * n_heads;
    const int grid = (int)(items < b200_num_sms() ? items : b200_num_sms());
    if (p.dbg) attn_fwd_tc05_kernel<true><<<grid, FWD_THREADS, SMEM_FWD_BYTES, stream>>>(tmQ, tmK, tmV, p);
    else attn_fwd_tc05_kernel<false><<<grid, FWD_THREADS, SMEM_FWD_BYTES, stream>>>(tmQ, tmK, tmV, p);
    B200_CHECK_LAUNCH("attn_causal_fwd_tc");
    return B200_OK;
}

// =============================================================================================
// backward on tcgen05: one CTA = one tile of 128 keys of one (batch, head), looping over the query tiles at or
// after the diagonal.  Five UMMA groups per query tile, all accumulators in TMEM (448 of 512 columns):
//   S^T  = K . Q_i^T        dP^T = V . dO_i^T       (two half tiles of 128 x 64, each in its own TMEM buffer, issued
//                                                    two pipeline units ahead of the math)
//   dV  += P^T . dO_i       dK  += dS^T . Q_i       (128 x 64, accumulated over the whole loop)
//   dQ_i = dS . K                                   (128 x 64 per tile; TMEM -> swizzled fp32 staging -> TMA reduce-add)
// P^T and dS^T are produced by two ping-pong groups of 8 math warps (group g = half g of every tile; thread = key row x
// 32 query columns), rounded to bf16 and written to 128B-swizzled shared memory where the UMMAs read them: K-major for
// dV / dK, and the same dS^T tile viewed MN-major as the A operand of dQ -- no transposes, no recomputation
// (5 matmuls, not 7).  DESIGN.md 3.1b has the measured history (1.01 ms mma.sync -> 0.41 ms).
// =============================================================================================
namespace {

constexpr int BWD_CWARPS = 16;                   // math warps: two groups of 8, thread = (key row, 32 of a half tile's 64 query columns)
constexpr int BWD_THREADS = 64 + 32 * BWD_CWARPS; // warp 0 TMA, warp 1 MMA, warps 2..17 compute
constexpr int SB_K = 0, SB_V = 16384;
constexpr int QS = 3;                            // (Q, dO) stages (4 measured no faster than 3; the 4th stage's 32 KB now stages dQ)
constexpr int SB_Q = 32768;                      // QS stages x (Q 16 KB + dO 16 KB)
constexpr int SB_P = SB_Q + QS * 32768;          // P^T : two 64-query atoms of [128 keys x 128 B]
constexpr int SB_DS = SB_P + 32768;              // dS^T: same layout
constexpr int SB_DQ = SB_DS + 32768;             // fp32 dQ tile for the TMA reduce: two 32-column boxes of [128 q x 128 B], 128B-swizzled
constexpr int SB_LSE = SB_DQ + 32768;            // float [2][2][128]: lse, delta per stage parity
constexpr int SB_BAR = SB_LSE + 2048;
constexpr int SMEM_BWD_BYTES = SB_BAR + 192;

// n_heads / Sq fill the slot between delta and dk: that keeps dv, dk_r, dv_r and rope_sin 16-byte aligned, and ptxas
// schedules the epilogue's parameter loads by that alignment
struct BwdParams {
    const float* lse;
    const float* delta;
    int n_heads, Sq;
    bf16* dk;
    bf16* dv;
    long long dk_b, dk_r, dv_b, dv_r;
    const bf16* rope_cos;        // optional fused RoPE backward on dK (dQ gets it in the finalize kernel)
    const bf16* rope_sin;
    int Sk;
    float scale;
};

// fp32 tile in shared memory += into global memory through the TMA unit (one instruction per 16 KB box instead of
// 1024 per-lane red.global instructions)
__device__ __forceinline__ void tma_reduce_add_3d(const CUtensorMap* tm, uint32_t smem_addr, int c0, int c1, int c2) {
    asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(tm), "r"(smem_addr), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// lse / delta of a group's 32 query columns reach its math warps through shared memory: one writer warp per column group
// stages the NEXT iteration's values before its pds_full arrival; the MMA thread issues S^T of that iteration only after all
// arrivals and the readers acquire s_full, so the hand-over is ordered by the mbarriers that are there anyway.
// compute-sanitizer's racecheck does not follow an ordering that passes through tcgen05.commit, so it reports these stores
// against the reads (profiles/r2_sanitizer_attention.txt).
__global__ void __launch_bounds__(BWD_THREADS, 1)
attn_bwd_tc05_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                     const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmdO,
                     const __grid_constant__ CUtensorMap tmDQ, const BwdParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SB_BAR);
    uint64_t* kv_full = bars + 0;
    uint64_t* q_full = bars + 1;      // [QS]
    uint64_t* q_empty = bars + 5;     // [QS]
    uint64_t* s_full = bars + 9;      // [2]  one per pipeline unit (half tile)
    uint64_t* pds_full = bars + 13;   // [2]
    uint64_t* dq_full = bars + 17;
    uint64_t* dq_empty = bars + 18;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 19);
    float* lse_s = reinterpret_cast<float*>(smem + SB_LSE);          // [2][128]
    float* delta_s = lse_s + 256;                                      // [2][128]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kt = blockIdx.y;       // slow grid index: all heavy (early-key) tiles are scheduled first
    const int bh = blockIdx.x;
    const int b = bh / p.n_heads, h = bh % p.n_heads;
    const int k0 = kt * BK;
    const int off = p.Sk - p.Sq;
    const int n_q = (p.Sq + BQ - 1) / BQ;
    int i0 = (k0 - off) / BQ;
    if (k0 - off < 0) i0 = 0;
    const int n_it = n_q - i0;                     // may be <= 0 when every query sits before this key tile

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmQ); prefetch_tmap(&tmK); prefetch_tmap(&tmV); prefetch_tmap(&tmdO);
        mbar_init(kv_full, 1);
        for (int s = 0; s < QS; s++) { mbar_init(&q_full[s], 1); mbar_init(&q_empty[s], 1); }
        for (int s = 0; s < 2; s++) { mbar_init(&s_full[s], 1); mbar_init(&pds_full[s], BWD_CWARPS / 2); }
        mbar_init(dq_full, 1); mbar_init(dq_empty, BWD_CWARPS / 2);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    if (warp >= 2 && (warp & 3) == 0) {
        // writer warps (row quarter 0): lse / delta of the first iteration, visible to everyone through the barrier below
        const int cw_ = warp - 2, qc_ = (cw_ >> 3) * 64 + ((cw_ >> 2) & 1) * 32;
        const int qi = i0 * BQ + qc_ + lane;
        const bool ok = n_it > 0 && qi < p.Sq;
        const long long rowb = ((long long)b * p.n_heads + h) * p.Sq;
        lse_s[qc_ + lane] = ok ? p.lse[rowb + qi] * LOG2E : 0.f;
        delta_s[qc_ + lane] = ok ? p.delta[rowb + qi] : 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // columns 0..255: two half-tile buffers, each S^T [128 keys x 64 q] | dP^T [128 x 64]
    const uint32_t tSB = tmem_base, tdV = tmem_base + 256, tdK = tmem_base + 320, tdQ = tmem_base + 384;

    if (warp == 0) {
        if (lane == 0) {
            mbar_expect_tx(kv_full, 2 * BK * D * 2);
            tma_load_3d(smem + SB_K, &tmK, kv_full, h * D, k0, b);
            tma_load_3d(smem + SB_V, &tmV, kv_full, h * D, k0, b);
            int stage = 0; uint32_t phase = 0;
            for (int it = 0; it < n_it; it++) {
                mbar_wait(&q_empty[stage], phase ^ 1);
                uint8_t* sQ = smem + SB_Q + stage * 32768;
                mbar_expect_tx(&q_full[stage], 2 * BQ * D * 2);
                tma_load_3d(sQ, &tmQ, &q_full[stage], h * D, (i0 + it) * BQ, b);
                tma_load_3d(sQ + 16384, &tmdO, &q_full[stage], h * D, (i0 + it) * BQ, b);
                if (++stage == QS) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && n_it > 0) {
            constexpr uint32_t id_s = make_idesc(128, 64, false, false);      // S^T, dP^T of one unit (64 queries)
            constexpr uint32_t id_kv = make_idesc(128, 64, false, true);      // dV, dK : A K-major (smem P^T/dS^T), B MN-major
            constexpr uint32_t id_dq = make_idesc(128, 64, true, true);       // dQ     : A = dS (MN-major view of dS^T), B = K MN-major
            const uint32_t sK = smem_u32(smem + SB_K), sV = smem_u32(smem + SB_V);
            const uint32_t sP = smem_u32(smem + SB_P), sDS = smem_u32(smem + SB_DS);
            mbar_wait(kv_full, 0);
            const uint64_t dKk = make_smem_desc(sK, 16, 1024), dVk = make_smem_desc(sV, 16, 1024);   // K-major A operands
            const uint64_t dKmn = make_smem_desc(sK, 16384, 1024);                                 // MN-major B of dQ
            const uint64_t dPk = make_smem_desc(sP, 16, 1024), dDSk = make_smem_desc(sDS, 16, 1024);
            const uint64_t dDSmn = make_smem_desc(sDS, 16384, 1024);
            // The pipeline unit is a half tile: 64 queries x 128 keys.  Unit u = (tile u/2, half u&1) owns TMEM buffer
            // u&1 and P^T/dS^T atom u&1, so S^T/dP^T of unit u+2 are produced while the math warps work on unit u+1
            // and the tensor pipe never sits on the critical path.
            const int n_units = 2 * n_it;
            auto issue_s = [&](int u) {
                const int it_ = u / 2, g = u % 2, st = it_ % QS;
                if (g == 0) mbar_wait(&q_full[st], (uint32_t)((it_ / QS) & 1));
                const uint32_t sQ = smem_u32(smem + SB_Q + st * 32768) + g * 8192;   // 64 query rows x 128 B
                const uint64_t dQk = make_smem_desc(sQ, 16, 1024), dOk = make_smem_desc(sQ + 16384, 16, 1024);
                const uint32_t tS = tSB + g * 128, tdP = tS + 64;
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < D / 16; k++) umma_f16(tS, desc_adv(dKk, k * 32), desc_adv(dQk, k * 32), id_s, k > 0);
#pragma unroll
                for (int k = 0; k < D / 16; k++) umma_f16(tdP, desc_adv(dVk, k * 32), desc_adv(dOk, k * 32), id_s, k > 0);
                umma_commit(&s_full[g]);
            };
#pragma unroll
            for (int u = 0; u < 2; u++)
                if (u < n_units) issue_s(u);
            for (int u = 0; u < n_units; u++) {
                const int it = u / 2, g = u % 2, st_cur = it % QS;
                const uint32_t sQ = smem_u32(smem + SB_Q + st_cur * 32768);
                const uint64_t dQmn = make_smem_desc(sQ, 16384, 1024), dOmn = make_smem_desc(sQ + 16384, 16384, 1024);
                mbar_wait(&pds_full[g], (uint32_t)(it & 1));    // P^T / dS^T columns of this unit written; its TMEM buffer is free
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < 4; k++) {                  // 16 query rows per step inside the half's 64-query atom
                    const int kk = g * 4 + k;
                    umma_f16(tdV, desc_adv(dPk, g * 16384 + k * 32), desc_adv(dOmn, kk * 2048), id_kv, (u > 0 || k > 0) ? 1u : 0u);
                }
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int kk = g * 4 + k;
                    umma_f16(tdK, desc_adv(dDSk, g * 16384 + k * 32), desc_adv(dQmn, kk * 2048), id_kv, (u > 0 || k > 0) ? 1u : 0u);
                }
                if (g == 1) {
                    mbar_wait(dq_empty, (uint32_t)((it & 1) ^ 1));      // previous dQ tile drained
                    tc_fence_after();
#pragma unroll
                    for (int kk = 0; kk < BK / 16; kk++)   // K dimension = keys: 16 key rows per step
                        umma_f16(tdQ, desc_adv(dDSmn, kk * 2048), desc_adv(dKmn, kk * 2048), id_dq, kk > 0);
                    umma_commit(dq_full);
                    umma_commit(&q_empty[st_cur]);
                }
                if (u + 2 < n_units) issue_s(u + 2);         // one tile ahead: not urgent, goes after this unit's dV/dK/dQ
            }
        }
    } else {
        // Two math groups of 8 warps: group g owns half g (64 queries) of every tile, i.e. every second pipeline unit,
        // with its own staging buffers and named barriers, so while one group waits (TMEM load, barrier, st.shared
        // + fence) the other is in its exp2/FMA stretch.  thread = (key row, 32 of the 64 query columns).
        const int cw = warp - 2;                       // 0..15
        const int quarter = warp & 3;
        const int hb = cw >> 3;                        // half tile == pipeline unit == math group of this warp
        const int cgi = (cw >> 2) & 1;                 // which 32 query columns of the half tile
        const int gtid = (cw & 7) * 32 + lane;         // 0..255 inside the group
        const int key_t = quarter * 32 + lane;         // key row inside the tile == TMEM lane
        const int key = k0 + key_t;
        const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
        const float sl2 = p.scale * LOG2E;
        const float* lse_g = p.lse + ((long long)b * p.n_heads + h) * p.Sq;
        const float* delta_g = p.delta + ((long long)b * p.n_heads + h) * p.Sq;
        const int qc0 = hb * 64 + cgi * 32;            // first query column (inside the tile) of this thread
        uint8_t* sP = smem + SB_P + hb * 16384 + key_t * 128;
        uint8_t* sDS = smem + SB_DS + hb * 16384 + key_t * 128;
        // lse / delta of this warp's 32 query columns (lane i -> column qc0 + i), fetched one iteration ahead by the writer warp
        // so the global load latency hides behind the previous iteration; the slot parity covers the one iteration two warps can
        // be apart (S_{it+1} of this half tile is issued only after all eight warps arrived on pds_full for it).
        auto fetch_ld = [&](int it_, float& lse_v, float& delta_v) {
            const int qi = (i0 + it_) * BQ + qc0 + lane;
            const bool ok = it_ < n_it && qi < p.Sq;
            lse_v = ok ? lse_g[qi] * LOG2E : 0.f;
            delta_v = ok ? delta_g[qi] : 0.f;
        };
        // dQ tile of a finished iteration, drained by group 0: TMEM lane = query row, this thread owns 32 columns
        auto drain_dq = [&](int q0_tile) {
            uint32_t r[32];
            tmem_ld32(tdQ + lane_addr + cgi * 32, r);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(dq_empty);                  // TMEM tile is free for the next dQ MMAs
            // the previous TMA reduce must have finished reading the staging tile before it is overwritten
            if (gtid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            asm volatile("bar.sync 1, 256;" ::: "memory");
            uint8_t* dst = smem + SB_DQ + cgi * 16384 + key_t * 128;
#pragma unroll
            for (int v = 0; v < 8; v++)
                *reinterpret_cast<uint4*>(dst + ((v ^ (key_t & 7)) << 4)) = make_uint4(r[4 * v], r[4 * v + 1], r[4 * v + 2], r[4 * v + 3]);
            fence_proxy_async_smem();
            asm volatile("bar.sync 3, 256;" ::: "memory");
            if (gtid == 0) {
                tma_reduce_add_3d(&tmDQ, smem_u32(smem + SB_DQ), h * D, q0_tile, b);
                tma_reduce_add_3d(&tmDQ, smem_u32(smem + SB_DQ + 16384), h * D + 32, q0_tile, b);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        };
        const bool drainer = hb == 0;
        float lse_next = 0.f, delta_next = 0.f;
        const bool writer = quarter == 0;
        for (int it = 0; it < n_it; it++) {
            const int q0 = (i0 + it) * BQ;
            if (writer) fetch_ld(it + 1, lse_next, delta_next);     // stored before this iteration's pds_full arrival
            const bool need_mask = (k0 + BK - 1 > q0 + off) || (k0 + BK > p.Sk) || (q0 + BQ > p.Sq);
            const float* lse_t = lse_s + (it & 1) * 128 + qc0;
            const float* delta_t = delta_s + (it & 1) * 128 + qc0;
            mbar_wait(&s_full[hb], (uint32_t)(it & 1));
            tc_fence_after();
            uint32_t pk[16], dk_[16];
#pragma unroll
            for (int hc = 0; hc < 2; hc++) {               // two chunks of 16 columns keep the register footprint flat
                uint32_t rs[16], rd[16];
                tmem_ld16(tSB + hb * 128 + lane_addr + cgi * 32 + hc * 16, rs);
                tmem_ld16(tSB + hb * 128 + 64 + lane_addr + cgi * 32 + hc * 16, rd);
                tmem_ld_wait();
                if (need_mask) {
                    // column c of this thread is visible iff key <= q0+qc0+c+off, key < Sk and q0+qc0+c < Sq
                    const int lo = (key < p.Sk) ? key - off - q0 - qc0 : 1 << 20;     // first visible column
                    const int hi = p.Sq - q0 - qc0;                                     // first column past the end
#pragma unroll
                    for (int i = 0; i < 16; i += 2) {
                        float pv[2], dsv[2];
#pragma unroll
                        for (int e = 0; e < 2; e++) {
                            const int qq = hc * 16 + i + e;
                            float pr = ex2_approx(fmaf(__uint_as_float(rs[i + e]), sl2, -lse_t[qq]));
                            if (qq < lo || qq >= hi) pr = 0.f;
                            pv[e] = pr;
                            dsv[e] = pr * (__uint_as_float(rd[i + e]) - delta_t[qq]);
                        }
                        pk[hc * 8 + (i >> 1)] = pack2(pv[0], pv[1]);
                        dk_[hc * 8 + (i >> 1)] = pack2(dsv[0], dsv[1]);
                    }
                    asm volatile("" ::: "memory");
                } else {
#pragma unroll
                    for (int i = 0; i < 16; i += 2) {
                        float pv[2], dsv[2];
#pragma unroll
                        for (int e = 0; e < 2; e++) {
                            const int qq = hc * 16 + i + e;
                            const float pr = ex2_approx(fmaf(__uint_as_float(rs[i + e]), sl2, -lse_t[qq]));
                            pv[e] = pr;
                            dsv[e] = pr * (__uint_as_float(rd[i + e]) - delta_t[qq]);
                        }
                        pk[hc * 8 + (i >> 1)] = pack2(pv[0], pv[1]);
                        dk_[hc * 8 + (i >> 1)] = pack2(dsv[0], dsv[1]);
                    }
                }
            }
            if (it > 0) {
                // the previous tile's dV / dK / dQ MMAs read both atoms: they must have retired before the overwrite
                mbar_wait(dq_full, (uint32_t)((it & 1) ^ 1));
                tc_fence_after();
            }
#pragma unroll
            for (int v = 0; v < 4; v++) {
                const int sw = ((cgi * 4 + v) ^ (key_t & 7)) << 4;
                *reinterpret_cast<uint4*>(sP + sw) = make_uint4(pk[4 * v], pk[4 * v + 1], pk[4 * v + 2], pk[4 * v + 3]);
                *reinterpret_cast<uint4*>(sDS + sw) = make_uint4(dk_[4 * v], dk_[4 * v + 1], dk_[4 * v + 2], dk_[4 * v + 3]);
            }
            if (writer && it + 1 < n_it) {
                lse_s[((it + 1) & 1) * 128 + qc0 + lane] = lse_next;
                delta_s[((it + 1) & 1) * 128 + qc0 + lane] = delta_next;
            }
            tc_fence_before();
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&pds_full[hb]);
            if (drainer && it > 0) drain_dq(q0 - BQ);   // off the critical path
        }
        if (n_it > 0) {
            mbar_wait(dq_full, (uint32_t)((n_it - 1) & 1));   // last tile's MMAs
            tc_fence_after();
            if (drainer) {
                drain_dq((i0 + n_it - 1) * BQ);
                if (gtid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            }
        }
        // epilogue: warps 2..9 write dK (two 16-column groups that form RoPE pairs d, d+32), warps 10..17 write dV
        // (32 columns each).  TMEM loads are warp-collective: every lane executes them, only the stores are predicated.
        {
            const int part = (cw >> 2) & 1;
            const bool is_dk = cw < 8;
            float v0[16], v1[16];
            if (n_it > 0) {
                uint32_t r[16];
                const uint32_t tsrc = (is_dk ? tdK : tdV) + lane_addr;
                const int c0 = is_dk ? part * 16 : part * 32, c1 = is_dk ? 32 + part * 16 : part * 32 + 16;
                tmem_ld16(tsrc + c0, r);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; i++) v0[i] = __uint_as_float(r[i]);
                tmem_ld16(tsrc + c1, r);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; i++) v1[i] = __uint_as_float(r[i]);
            } else {
#pragma unroll
                for (int i = 0; i < 16; i++) { v0[i] = 0.f; v1[i] = 0.f; }
            }
            if (key < p.Sk) {
                if (is_dk) {
#pragma unroll
                    for (int i = 0; i < 16; i++) { v0[i] *= p.scale; v1[i] *= p.scale; }
                    if (p.rope_cos) {
                        const bf16* cp = p.rope_cos + (size_t)key * 32 + part * 16;
                        const bf16* sp = p.rope_sin + (size_t)key * 32 + part * 16;
#pragma unroll
                        for (int i = 0; i < 16; i++) {
                            const float c = __bfloat162float(cp[i]), sn = __bfloat162float(sp[i]);
                            const float a = v0[i], bb = v1[i];
                            v0[i] = a * c + bb * sn;
                            v1[i] = bb * c - a * sn;
                        }
                    }
                    bf16* d0 = p.dk + b * p.dk_b + (long long)key * p.dk_r + h * D + part * 16;
                    *reinterpret_cast<uint4*>(d0) = pack8(v0);
                    *reinterpret_cast<uint4*>(d0 + 8) = pack8(v0 + 8);
                    *reinterpret_cast<uint4*>(d0 + 32) = pack8(v1);
                    *reinterpret_cast<uint4*>(d0 + 40) = pack8(v1 + 8);
                } else {
                    bf16* d0 = p.dv + b * p.dv_b + (long long)key * p.dv_r + h * D + part * 32;
                    *reinterpret_cast<uint4*>(d0) = pack8(v0);
                    *reinterpret_cast<uint4*>(d0 + 8) = pack8(v0 + 8);
                    *reinterpret_cast<uint4*>(d0 + 16) = pack8(v1);
                    *reinterpret_cast<uint4*>(d0 + 24) = pack8(v1 + 8);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// dq[rows, heads*64] (bf16, row pitch ld) = scale * (optional RoPE^T) dq_acc (fp32)
__global__ void attn_bwd_dq_finalize_kernel(const float* __restrict__ acc, bf16* __restrict__ dq, long long rows, int W, int ld,
                                            int S, float scale, const bf16* __restrict__ rope_cos,
                                            const bf16* __restrict__ rope_sin) {
    B200_PDL_TRIGGER();
    // one thread = 8 columns d0..d0+7 of the first half of a head and the matching 8 of the second half
    const long long n = rows * (W / 16);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / (W / 16);
        const int u = (int)(i % (W / 16));
        const int hd = u >> 2, d0 = (u & 3) * 8;
        const float* src = acc + r * W + hd * 64 + d0;
        float a[8], bq[8];
#pragma unroll
        for (int j = 0; j < 8; j++) { a[j] = src[j] * scale; bq[j] = src[32 + j] * scale; }
        if (rope_cos) {
            const int pos = (int)(r % S);
            float c[8], s[8];
            unpack8(*reinterpret_cast<const uint4*>(rope_cos + (size_t)pos * 32 + d0), c);
            unpack8(*reinterpret_cast<const uint4*>(rope_sin + (size_t)pos * 32 + d0), s);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const float x = a[j], y = bq[j];
                a[j] = x * c[j] + y * s[j];
                bq[j] = y * c[j] - x * s[j];
            }
        }
        bf16* dst = dq + r * ld + hd * 64 + d0;
        *reinterpret_cast<uint4*>(dst) = pack8(a);
        *reinterpret_cast<uint4*>(dst + 32) = pack8(bq);
    }
}

}   // namespace

// tuning hook: device buffer of 128 int64 receiving the per-phase cycle sums of the forward kernel's softmax warps (NULL = off)
extern "C" void b200_attn_debug_trace(long long* buf) { g_attn_dbg = buf; }

// defined in attn_flash.cu
int b200_attn_bwd_delta_launch(const void* o, const void* d_o, float* delta, const long long* so, const long long* sdo,
                               int batch, int n_heads, int Sq, cudaStream_t stream);

extern "C" size_t b200_attn_causal_bwd_tc_workspace_bytes(int batch, int n_heads, int Sq) {
    return (size_t)batch * Sq * n_heads * D * sizeof(float) + (size_t)batch * n_heads * Sq * sizeof(float);
}

// Same contract as b200_attn_causal_bwd; workspace = fp32 dQ accumulator + delta (b200_attn_causal_bwd_tc_workspace_bytes).
// q/k/v/dq/dk/dv are thirds of packed [batch*S, ld] activations with heads as contiguous 64-column blocks.
extern "C" int b200_attn_causal_bwd_tc(const void* q, const void* k, const void* v, const void* o, const void* d_o,
                                       const float* lse, void* dq, void* dk, void* dv,
                                       const long long* strides /* 8 x {b,r,h}: q,k,v,o,do,dq,dk,dv */, int batch,
                                       int n_heads, int Sq, int Sk, int head_dim, float scale, const void* rope_cos,
                                       const void* rope_sin, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    B200_CHECK_ARG(head_dim == D, "attn_causal_bwd_tc: head_dim %d unsupported (64 only)", head_dim);
    B200_CHECK_ARG(Sk == Sq, "attn_causal_bwd_tc: training shapes only (Sk == Sq)");
    B200_CHECK_ARG(n_heads % 4 == 0, "attn_causal_bwd_tc: n_heads must be a multiple of 4");
    for (int i = 0; i < 8; i++)
        B200_CHECK_ARG(strides[3 * i + 2] == D, "attn_causal_bwd_tc: heads must be contiguous blocks of 64 columns");
    B200_CHECK_ARG(strides[15] == (long long)Sq * strides[16], "attn_causal_bwd_tc: dq batches must be contiguous");
    B200_CHECK_ARG(workspace_bytes >= b200_attn_causal_bwd_tc_workspace_bytes(batch, n_heads, Sq),
                   "attn_causal_bwd_tc: workspace too small");
    if (batch == 0 || Sq == 0) return B200_OK;
    const long long W = (long long)n_heads * D;
    float* dq_acc = (float*)workspace;
    float* delta = dq_acc + (size_t)batch * Sq * W;
    {   // delta = rowsum(dO * O), shared with the mma.sync path
        int rc = b200_attn_bwd_delta_launch(o, d_o, delta, strides + 9, strides + 12, batch, n_heads, Sq, stream);
        if (rc) return rc;
    }
    CUtensorMap tmQ, tmK, tmV, tmdO;
    int rc;
    if ((rc = tc05_make_tmap_3d(&tmQ, q, W, Sq, batch, strides[1], strides[0], D, BQ))) return rc;
    if ((rc = tc05_make_tmap_3d(&tmK, k, W, Sk, batch, strides[4], strides[3], D, BK))) return rc;
    if ((rc = tc05_make_tmap_3d(&tmV, v, W, Sk, batch, strides[7], strides[6], D, BK))) return rc;
    if ((rc = tc05_make_tmap_3d(&tmdO, d_o, W, Sq, batch, strides[13], strides[12], D, BQ))) return rc;
    CUtensorMap tmDQ;
    if ((rc = tc05_make_tmap_3d_f32(&tmDQ, dq_acc, W, Sq, batch, W, (long long)Sq * W, 32, BQ))) return rc;
    BwdParams p;
    p.lse = lse; p.delta = delta;
    p.dk = (bf16*)dk; p.dv = (bf16*)dv;
    p.dk_b = strides[18]; p.dk_r = strides[19]; p.dv_b = strides[21]; p.dv_r = strides[22];
    p.rope_cos = (const bf16*)rope_cos; p.rope_sin = (const bf16*)rope_sin;
    p.n_heads = n_heads; p.Sq = Sq; p.Sk = Sk; p.scale = scale;
    static bool configured = false;
    if (!configured) {
        B200_CUDA(cudaFuncSetAttribute(attn_bwd_tc05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BWD_BYTES), "attn_bwd_tc smem");
        configured = true;
    }
    B200_CUDA(cudaMemsetAsync(dq_acc, 0, (size_t)batch * Sq * W * sizeof(float), stream), "attn_bwd_tc memset");
    dim3 grid(batch * n_heads, (Sk + BK - 1) / BK);   // tiles on the slow index: longest first across all heads
    attn_bwd_tc05_kernel<<<grid, BWD_THREADS, SMEM_BWD_BYTES, stream>>>(tmQ, tmK, tmV, tmdO, tmDQ, p);
    B200_CHECK_LAUNCH("attn_causal_bwd_tc");
    const long long rows = (long long)batch * Sq;
    long long nthr = rows * (W / 16);
    int blocks = (int)((nthr + 255) / 256);
    if (blocks > b200_num_sms() * 16) blocks = b200_num_sms() * 16;
    attn_bwd_dq_finalize_kernel<<<blocks, 256, 0, stream>>>(dq_acc, (bf16*)dq, rows, (int)W, (int)strides[16], Sq, scale,
                                                            (const bf16*)rope_cos, (const bf16*)rope_sin);
    B200_CHECK_LAUNCH("attn_bwd_dq_finalize");
    return B200_OK;
}
