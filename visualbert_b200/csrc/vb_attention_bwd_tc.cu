// vb_attention_bwd_tc.cu — attention backward on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), seq <= 192.
//
// Adjoint of reference modeling.py:241-256 (QK^T / sqrt(d) + mask -> softmax -> dropout -> P V). One persistent CTA per SM
// walks over (batch, head) items. All five contractions run on tcgen05.mma with TMEM accumulators; the element-wise
// work runs TRANSPOSED — TMEM lane = key, column = query — so nothing needs a cross-thread reduction (the row
// statistics lse[q] and D[q] = sum_d dO O are per COLUMN vectors staged in shared memory).
//
// Work unit = (key tile kt of 128 lanes, block qb of 64 queries); the second key tile of seq = 128 + r sits at a rotating
// lane offset (see vb_attention_tc.cu). Unit g of the CTA's sequence belongs to element-wise warp-group g % 2 and to
// TMEM slot g % 2, so the MMAs of one unit run under the element-wise pass of the other:
//     S^T  = K_kt Q_qb^T     M=128 N=64 K=64     -> slot columns  0..63
//     dP^T = V_kt dO_qb^T    M=128 N=64 K=64     -> slot columns 64..127
//     element-wise (4 warps, thread = key row):
//         p   = exp2(s * scale*log2e + mask[key] - lse[q])
//         Pd  = keep ? p / (1-pd) : 0               -> bf16 -> TMEM, in place over the consumed S^T columns
//         dS  = p * (keep ? dP / (1-pd) : 0 - D[q]) -> bf16 -> shared memory [key][q], 128B-swizzled 64-query atom
//     dV_kt += Pd^T dO_qb    M=128 N=64 K=64     A = Pd^T FROM TMEM,  B = dO rows (MN-major)        -> TMEM (per kt)
//     dK_kt += dS^T Q_qb     M=128 N=64 K=64     A = dS^T FROM TMEM (second in-place copy, over dP^T), B = Q rows (MN-major)
//     dQ_m  += dS K_kt       M=128 (queries of tile m = atoms 2m, 2m+1) N=64 K=keys of kt
//                            A = the SAME dS^T bytes read MN-major, B = K (MN-major)                  -> TMEM (per item)
// TMEM (512 columns): slot 0 | slot 1 | dV dK | dQ tile 0, tile 1. The warp-group that finishes a key tile's last unit
// drains dV / dK (lane = key), the one that finishes the item's last unit drains dQ (lane = query).
//
//   warp 0  TMA producer (Q, dO, K double-buffered per item; V single-buffered: it is dead after the last dP^T MMA)
//   warp 1  MMA issuer (one thread)      warp 2  TMEM allocator      warp 3  stages lse * log2e and D of the item
//   warps 4-7 / 8-11  element-wise warp-groups 0 / 1 (+ output drains)
#include "vb_attention.cuh"

namespace vb {

namespace {

constexpr int kRows = 128;            // UMMA M (keys per tile / queries per dQ tile)
constexpr int kWgT = 128;             // threads per warp-group
constexpr int kThreadsBw = 128 + 2 * kWgT;
constexpr int kMaxNpq = 192;
constexpr uint32_t kTmSlot = 128, kTmAcc = 256, kTmDq = 384;   // TMEM columns: slot s at 128 s (S^T | dP^T), dV, dK, dQ tiles

__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ uint32_t idesc_bw(int m, int n, bool a_mn, bool b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn) << 15) | (static_cast<uint32_t>(b_mn) << 16) |
           (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

struct BwLayout {   // byte offsets from the 1 KB-aligned base
    int qbytes;      // npq * 128 (Q and dO tiles)
    int k1bytes;     // r2pad * 128 (compact window of the second key tile)
    int stage_bytes; // Q | dO | K0
    int nstage;
    int k1_off;      // [nstage] K windows, then the V window, then dS^T of the second tile (natoms x k1bytes)
    int v1_off, ds1_off;
    int ds0_off;     // natoms x 16 KB
    int v0_off;
    int vec_off;     // fp32 [nstage][2][kMaxNpq]: lse * log2e | D
    int bar_off, tmem_ptr_off, total;
};
__host__ __device__ inline BwLayout bw_layout(int npq, int r2pad, int nstage) {
    BwLayout L;
    const int natoms = (npq + 63) / 64;
    L.qbytes = npq * 128;
    L.k1bytes = r2pad * 128;
    L.stage_bytes = 2 * L.qbytes + kRows * 128;
    L.nstage = nstage;
    L.k1_off = nstage * L.stage_bytes;
    L.v1_off = L.k1_off + nstage * L.k1bytes;
    L.ds1_off = L.v1_off + L.k1bytes;
    L.ds0_off = L.ds1_off + natoms * L.k1bytes;
    L.v0_off = L.ds0_off + natoms * kRows * 128;
    L.vec_off = L.v0_off + kRows * 128;
    L.bar_off = L.vec_off + nstage * 2 * kMaxNpq * 4;
    L.tmem_ptr_off = L.bar_off + 16 * 8;
    L.total = L.tmem_ptr_off + 16 + 1024;
    return L;
}

struct BwParams {
    AttnParams a;
    int npq;     // queries padded to 16 (MMA N of S^T / dP^T, K of dV / dK)
    int nqb;     // 64-query blocks per key tile
    int nkt;     // key tiles (1 or 2)
    int r2;      // keys of the second tile, r2pad = r2 rounded up to 16
    int r2pad;
    int nkb;     // ceil(S / 64)
    int nstage;
    long long* dbg;   // optional clock64 stamps of CTA 0 (VB_TC_DEBUG=1): [unit < 48][8]
};

__device__ __forceinline__ int kt1_offset(int li, int r2pad) {
    const int lim = kRows - r2pad;   // multiple of 16
    const int o = (li & 3) * 32;
    return o < lim ? o : lim;
}

__global__ void __launch_bounds__(kThreadsBw, 1)
attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO,
                   const __grid_constant__ CUtensorMap tmK0, const __grid_constant__ CUtensorMap tmK1, const BwParams bp) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base - raw);
    const AttnParams& p = bp.a;
    const BwLayout L = bw_layout(bp.npq, bp.r2pad, bp.nstage);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int S = p.S, npq = bp.npq, nkt = bp.nkt, nstage = bp.nstage;

    auto q_tile = [&](int s) { return base + s * L.stage_bytes; };
    auto do_tile = [&](int s) { return base + s * L.stage_bytes + L.qbytes; };
    auto k0_tile = [&](int s) { return base + s * L.stage_bytes + 2 * L.qbytes; };
    auto k1_win = [&](int s) { return base + L.k1_off + s * L.k1bytes; };
    const uint32_t v0_tile = base + L.v0_off, v1_win = base + L.v1_off;
    const uint32_t ds0 = base + L.ds0_off, ds1 = base + L.ds1_off;
    auto bar = [&](int i) { return base + L.bar_off + 8 * i; };
    enum { IN_FULL0 = 0, IN_EMPTY0 = 2, V_FULL = 4, V_EMPTY = 5, SD_FULL0 = 6, EW_DONE0 = 8, ACC_FULL = 10, ACC_EMPTY = 11, DQ_FULL = 12,
           DQ_EMPTY = 13 };
    volatile uint32_t* tmem_ptr = reinterpret_cast<volatile uint32_t*>(smem + L.tmem_ptr_off);
    float* svec_all = reinterpret_cast<float*>(smem + L.vec_off);

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmQ);
        tma_prefetch_desc(&tmDO);
        tma_prefetch_desc(&tmK0);
        tma_prefetch_desc(&tmK1);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar(IN_FULL0 + s), 2);   // TMA producer (expect_tx) + the vector stager
            mbar_init(bar(IN_EMPTY0 + s), 1);
        }
        mbar_init(bar(V_FULL), 1);
        mbar_init(bar(V_EMPTY), 1);
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar(SD_FULL0 + s), 1);
            mbar_init(bar(EW_DONE0 + s), kWgT);
        }
        mbar_init(bar(ACC_FULL), 1);
        mbar_init(bar(ACC_EMPTY), kWgT);   // the warp-group that drains dV / dK
        mbar_init(bar(DQ_FULL), 1);
        mbar_init(bar(DQ_EMPTY), kWgT);
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc(base + L.tmem_ptr_off, 512);
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    pdl_trigger();
    pdl_wait();

    const int total = p.B * p.A;
    const int n_local = (total - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);

    // register split: 128 x 88 (control warpgroup) + 256 x 208 (element-wise warpgroups) = the 384 x 168 of the launch
    const int nqb = bp.nqb;
    const int upi = nkt * nqb;              // units per item, ordered kt-major
    const int n_units = n_local * upi;      // units of this CTA
    if (warp < 4) {
        reg_dec<88>();
        if (warp == 0) {
            if (lane == 0) {
                // ---------------- TMA producer ----------------
                const uint32_t in_tx = static_cast<uint32_t>(2 * npq * 128 + kRows * 128 + (nkt == 2 ? bp.r2pad * 128 : 0));
                const uint32_t v_tx = static_cast<uint32_t>(kRows * 128 + (nkt == 2 ? bp.r2pad * 128 : 0));
                for (int li = 0; li < n_local; ++li) {
                    const int item = blockIdx.x + li * gridDim.x;
                    const int b = item / p.A, h = item % p.A;
                    const int s = li % nstage;
                    mbar_wait(bar(IN_EMPTY0 + s), ((li / nstage) & 1) ^ 1u);
                    mbar_arrive_expect_tx(bar(IN_FULL0 + s), in_tx);
                    tma_load_3d(q_tile(s), &tmQ, bar(IN_FULL0 + s), h * kHd, 0, b);
                    tma_load_3d(do_tile(s), &tmDO, bar(IN_FULL0 + s), h * kHd, 0, b);
                    tma_load_3d(k0_tile(s), &tmK0, bar(IN_FULL0 + s), p.H + h * kHd, 0, b);
                    if (nkt == 2) tma_load_3d(k1_win(s), &tmK1, bar(IN_FULL0 + s), p.H + h * kHd, kRows, b);
                    mbar_wait(bar(V_EMPTY), (li & 1) ^ 1u);
                    mbar_arrive_expect_tx(bar(V_FULL), v_tx);
                    tma_load_3d(v0_tile, &tmK0, bar(V_FULL), 2 * p.H + h * kHd, 0, b);
                    if (nkt == 2) tma_load_3d(v1_win, &tmK1, bar(V_FULL), 2 * p.H + h * kHd, kRows, b);
                }
            }
        } else if (warp == 1) {
            {
                // ---------------- MMA issuer: the whole warp runs the loop converged, one elected lane issues ----------------
                // ONE copy of every MMA sequence; per MMA a 32-bit add per descriptor and the tcgen05.mma itself (the issuing
                // thread's instruction stream is the critical path of the pipeline).
                const uint32_t idesc_vk = idesc_bw(kRows, kHd, false, true);
                const uint32_t idesc_dq = idesc_bw(kRows, kHd, true, true);
                const uint32_t tm_acc = tmem_base + kTmAcc, tm_dq = tmem_base + kTmDq;
                int next_sd = 0;   // next unit whose S^T / dP^T have not been issued yet
                for (int g = -1; g < n_units; ++g) {
                    bool item_end = false;
                    int li_g = 0;
                    if (g >= 0) {
                        const int li = g / upi, ul = g - li * upi, kt = ul / nqb, qb = ul - kt * nqb;
                        const int s = li % nstage, slot = g & 1;
                        const int bw = min(64, npq - 64 * qb);
                        const uint32_t off = kt == 0 ? 0u : static_cast<uint32_t>(kt1_offset(li, bp.r2pad) * 128);
                        const uint32_t ds_base = kt == 0 ? ds0 : ds1;
                        const uint32_t ds_atom = kt == 0 ? kRows * 128 : static_cast<uint32_t>(L.k1bytes);
                        li_g = li;
                        item_end = ul == upi - 1;
                        const bool stamp = bp.dbg != nullptr && blockIdx.x == 0 && g < 48 && lane == 0;
                        if (stamp) bp.dbg[g * 8 + 4] = clock64();
                        mbar_wait(bar(EW_DONE0 + slot), (g >> 1) & 1);
                        if (stamp) bp.dbg[g * 8 + 5] = clock64();
                        if (qb == 0) mbar_wait(bar(ACC_EMPTY), ((li * nkt + kt) & 1) ^ 1u);   // dV / dK of the previous key tile drained
                        tcgen05_fence_after();
                        const UmmaDesc d_do = make_umma_desc_sw128(do_tile(s) + qb * 8192, 0, 1024);
                        const UmmaDesc d_q = make_umma_desc_sw128(q_tile(s) + qb * 8192, 0, 1024);
                        const uint32_t tm_pd = tmem_base + slot * kTmSlot;
                        const bool first_dq = ((qb & 1) || qb == nqb - 1) && kt == 0 && (qb >> 1) == 0;
                        if (first_dq) {   // first dQ MMA of the item: the previous item's dQ must be drained
                            mbar_wait(bar(DQ_EMPTY), (li & 1) ^ 1u);
                            tcgen05_fence_after();
                        }
                        if (elect_one()) {
                        // dV_kt += Pd^T dO_qb (A from TMEM, 8 columns per k-step), dK_kt += dS^T Q_qb (A = this unit's dS^T atom)
                        for (int k = 0; k < bw / 16; ++k)
                            umma_bf16_ts(tm_acc, tm_pd + k * 8, d_do.at(k * 2048), idesc_vk, (qb > 0 || k > 0) ? 1u : 0u);
                        for (int k = 0; k < bw / 16; ++k)
                            umma_bf16_ts(tm_acc + kHd, tm_pd + 64 + k * 8, d_q.at(k * 2048), idesc_vk, (qb > 0 || k > 0) ? 1u : 0u);
                        // dQ tile m (queries of atoms 2m, 2m+1) += dS K_kt once both of its atoms hold this key tile's dS^T
                        if ((qb & 1) || qb == nqb - 1) {
                            const int m = qb >> 1;
                            const UmmaDesc a_ds = make_umma_desc_sw128(ds_base + (2 * m) * ds_atom, ds_atom, 1024);
                            const UmmaDesc d_k = make_umma_desc_sw128(kt == 0 ? k0_tile(s) : k1_win(s), 0, 1024);
                            const int jsteps = kt == 0 ? kRows / 16 : bp.r2pad / 16;   // 16 key rows = 2048 B per step
                            for (int j = 0; j < jsteps; ++j)
                                umma_bf16(tm_dq + m * kHd, a_ds.at(j * 2048), d_k.at(j * 2048), idesc_dq, (kt > 0 || j > 0) ? 1u : 0u);
                        }
                        if (qb == nqb - 1) umma_commit(bar(ACC_FULL));
                        if (item_end) {
                            umma_commit(bar(DQ_FULL));
                            umma_commit(bar(IN_EMPTY0 + s));   // every MMA of the item has retired: Q / dO / K are free
                        }
                        }
                        __syncwarp();
                        if (stamp) bp.dbg[g * 8 + 6] = clock64();
                    }
                    // S^T / dP^T of the units up to g + 2 (a unit's slot is free once dV of the unit two before it is issued);
                    // with a single input stage the next item's first units wait until this item has released the inputs
                    while (next_sd < n_units && next_sd <= g + 2) {
                        const int li = next_sd / upi, ul = next_sd - li * upi, kt = ul / nqb, qb = ul - kt * nqb;
                        if (nstage == 1 && li > (g < 0 ? 0 : li_g + (item_end ? 1 : 0))) break;   // its inputs are not released yet
                        // its element-wise pass overwrites dS^T atom qb of tile kt, which the previous item's dQ MMA reads at
                        // unit (qb | 1) or nqb - 1 of that tile: issue after that MMA, so SD_FULL (in-order completion) also
                        // means the atom is free.
                        // Binds only with one or two units per item (S <= 128); it also keeps the shared ACC_FULL / DQ_FULL
                        // waits of the two warp-groups in phase order when every item has a single unit.
                        if (next_sd - upi + min(qb | 1, nqb - 1) - qb > g) break;
                        const int s = li % nstage, slot = next_sd & 1;
                        const int bw = min(64, npq - 64 * qb);
                        if (ul == 0) {
                            mbar_wait(bar(IN_FULL0 + s), (li / nstage) & 1);
                            mbar_wait(bar(V_FULL), li & 1);
                            tcgen05_fence_after();
                        }
                        const uint32_t off = kt == 0 ? 0u : static_cast<uint32_t>(kt1_offset(li, bp.r2pad) * 128);
                        const UmmaDesc d_k = make_umma_desc_sw128(kt == 0 ? k0_tile(s) : k1_win(s) - off, 0, 1024);
                        const UmmaDesc d_v = make_umma_desc_sw128(kt == 0 ? v0_tile : v1_win - off, 0, 1024);
                        const UmmaDesc d_q = make_umma_desc_sw128(q_tile(s) + qb * 8192, 0, 1024);
                        const UmmaDesc d_do = make_umma_desc_sw128(do_tile(s) + qb * 8192, 0, 1024);
                        const uint32_t idesc_sd = idesc_bw(kRows, bw, false, false);
                        const uint32_t tm_slot = tmem_base + slot * kTmSlot;
                        if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < kHd / 16; ++k) umma_bf16(tm_slot, d_k.at(k * 32), d_q.at(k * 32), idesc_sd, k > 0 ? 1u : 0u);
#pragma unroll
                        for (int k = 0; k < kHd / 16; ++k) umma_bf16(tm_slot + 64, d_v.at(k * 32), d_do.at(k * 32), idesc_sd, k > 0 ? 1u : 0u);
                        umma_commit(bar(SD_FULL0 + slot));
                        if (ul == upi - 1) umma_commit(bar(V_EMPTY));   // V is dead once the item's last dP^T has retired
                        }
                        __syncwarp();
                        if (bp.dbg != nullptr && blockIdx.x == 0 && next_sd < 48 && lane == 0) bp.dbg[next_sd * 8 + 7] = clock64();
                        ++next_sd;
                    }
                }
            }
        } else if (warp == 3) {
            // ---------------- per-item column vectors: lse * log2e (+inf on padding: p = 0) and D ----------------
            for (int li = 0; li < n_local; ++li) {
                const int item = blockIdx.x + li * gridDim.x;
                const int s = li % nstage;
                mbar_wait(bar(IN_EMPTY0 + s), ((li / nstage) & 1) ^ 1u);
                float* sv = svec_all + s * 2 * kMaxNpq;
                const float* lsep = p.lse + static_cast<long long>(item) * S;
                const float* drp = p.drow + static_cast<long long>(item) * S;
                for (int i = lane; i < npq; i += 32) {
                    sv[i] = i < S ? __ldg(lsep + i) * kLog2e : INFINITY;
                    sv[kMaxNpq + i] = i < S ? __ldg(drp + i) : 0.f;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(bar(IN_FULL0 + s));
            }
        }
    } else {
        reg_inc<208>();
        // ---------------- element-wise + drains: warp-group wg owns the units g = wg, wg + 2, ... and TMEM slot wg ----------------
        const int wg = (warp - 4) >> 2;
        const int q4 = warp & 3;
        const int r = q4 * 32 + lane;                       // TMEM lane of this thread
        const uint32_t lane_sel = static_cast<uint32_t>(q4 * 32) << 16;
        const float sc2 = p.scale * kLog2e;
        const bool drop = p.drop_scale != 0.f;
        const float ds = drop ? p.drop_scale : 1.f;
        const int np64 = bp.nkb * kBlk;
        const uint32_t tm_st = tmem_base + wg * kTmSlot + lane_sel, tm_dpt = tm_st + 64;
        const uint32_t tm_acc = tmem_base + kTmAcc + lane_sel, tm_dq = tmem_base + kTmDq + lane_sel;
        const unsigned long long* keepT = p.keep + static_cast<long long>(p.B) * p.A * np64 * bp.nkb;
        const long long ld3 = 3LL * p.H;
        // 64 fp32 TMEM columns of this thread's lane -> * mul -> bf16 -> 128 contiguous bytes of global memory
        auto drain64 = [&](uint32_t tm, bf16* dst, float mul, bool valid, bool wload) {
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                uint32_t o[2][16];
                if (wload) {
                    tmem_ld_32x32b_x16(tm + half * 32, o[0]);
                    tmem_ld_32x32b_x16(tm + half * 32 + 16, o[1]);
                    tmem_ld_wait();
                }
                if (valid) {
#pragma unroll
                    for (int jj = 0; jj < 2; ++jj) {
                        uint32_t w[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            w[i] = pack_bf16x2(__uint_as_float(o[jj][2 * i]) * mul, __uint_as_float(o[jj][2 * i + 1]) * mul);
                        stg_v8(dst + half * 32 + jj * 16, w);
                    }
                }
            }
        };
        for (int g = wg; g < n_units; g += 2) {
            const int li = g / upi, ul = g - li * upi, kt = ul / nqb, qb = ul - kt * nqb;
            const int item = blockIdx.x + li * gridDim.x;
            const int b = item / p.A, h = item % p.A;
            const int s = li % nstage;
            const float* slse = svec_all + s * 2 * kMaxNpq + qb * 64;
            const float* sD = slse + kMaxNpq;
            bf16* dbase = p.dqkv + static_cast<long long>(b) * S * ld3 + h * kHd;
            const int off = kt == 0 ? 0 : kt1_offset(li, bp.r2pad);
            const int wrows = kt == 0 ? kRows : bp.r2pad;            // rows of this tile that carry (possibly zero) data
            const bool inwin = r >= off && r < off + wrows;
            const bool wany = __any_sync(0xffffffffu, inwin);
            const int j = kt * kRows + r - off;                      // key index of this lane
            const int np8 = min(64, npq - 64 * qb) / 8;              // 8-query pieces of this unit (even)
            float bias2 = -INFINITY;
            unsigned long long kw = ~0ull;
            if (inwin && j < S) {
                bias2 = __ldg(p.mask_bias + static_cast<long long>(b) * S + j) * kLog2e;
                if (drop) kw = keepT[(static_cast<long long>(item) * np64 + j) * bp.nkb + qb];   // 64 queries of this key
            }
            const bool stamp = bp.dbg != nullptr && blockIdx.x == 0 && (threadIdx.x & 127) == 0 && g < 48;
            if (stamp) bp.dbg[g * 8 + 0] = clock64();
            mbar_wait(bar(IN_FULL0 + s), (li / nstage) & 1);   // lse / D of this item staged and visible
            mbar_wait(bar(SD_FULL0 + wg), (g >> 1) & 1);
            tcgen05_fence_after();
            if (stamp) bp.dbg[g * 8 + 1] = clock64();
            if (wany) {
                // dS^T row of this lane inside the unit's 64-query atom: 16-byte chunks XOR-swizzled with (row & 7)
                const uint32_t ds_row = kt == 0 ? ds0 + qb * (kRows * 128) + r * 128 : ds1 + qb * L.k1bytes + (r - off) * 128;
                const int sw = r & 7;
                auto ew8 = [&](const uint32_t (&vs)[8], const uint32_t (&vd)[8], int i) {
                    const float4* l4 = reinterpret_cast<const float4*>(slse + i * 8);
                    const float4* d4 = reinterpret_cast<const float4*>(sD + i * 8);
                    const uint32_t bits = drop ? static_cast<uint32_t>(kw >> (i * 8)) : 0xffu;
                    float pd[8], dsv[8];
#pragma unroll
                    for (int jj = 0; jj < 2; ++jj) {
                        const float4 ll = l4[jj], dd = d4[jj];
                        const float lv[4] = {ll.x, ll.y, ll.z, ll.w}, dv[4] = {dd.x, dd.y, dd.z, dd.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int k = 4 * jj + e;
                            const float pr = fast_ex2(fmaf(__uint_as_float(vs[k]), sc2, bias2) - lv[e]);
                            const float t = ((bits >> k) & 1u) ? ds : 0.f;
                            pd[k] = pr * t;
                            dsv[k] = pr * fmaf(__uint_as_float(vd[k]), t, -dv[e]);
                        }
                    }
                    // Pd^T: 4 columns inside this thread's consumed S^T columns (8 bf16)
                    tmem_st_32x32b_x4(tm_st + i * 4, pack_bf16x2(pd[0], pd[1]), pack_bf16x2(pd[2], pd[3]), pack_bf16x2(pd[4], pd[5]),
                                      pack_bf16x2(pd[6], pd[7]));
                    // dS^T twice: in TMEM (in place over the consumed dP^T columns) as the A operand of dK — an MMA whose A comes
                    // from TMEM skips the 4 KB shared-memory operand read (measured 40 vs 69 cycles at N = 64, scripts/micro/
                    // umma_rate.cu) — and in shared memory, where the dQ MMA reads the same bytes MN-major
                    const uint32_t s0 = pack_bf16x2(dsv[0], dsv[1]), s1 = pack_bf16x2(dsv[2], dsv[3]), s2 = pack_bf16x2(dsv[4], dsv[5]),
                                   s3 = pack_bf16x2(dsv[6], dsv[7]);
                    tmem_st_32x32b_x4(tm_dpt + i * 4, s0, s1, s2, s3);
                    if (inwin) st_shared_v4(ds_row + ((i ^ sw) << 4), s0, s1, s2, s3);
                };
                uint32_t sa[8], da[8], sb[8], db[8];
                tmem_ld_32x32b_x8(tm_st, sa);
                tmem_ld_32x32b_x8(tm_dpt, da);
                for (int i = 0; i < np8; i += 2) {
                    tmem_ld_wait();
                    tmem_ld_32x32b_x8(tm_st + (i + 1) * 8, sb);
                    tmem_ld_32x32b_x8(tm_dpt + (i + 1) * 8, db);
                    ew8(sa, da, i);
                    tmem_ld_wait();
                    if (i + 2 < np8) {
                        tmem_ld_32x32b_x8(tm_st + (i + 2) * 8, sa);
                        tmem_ld_32x32b_x8(tm_dpt + (i + 2) * 8, da);
                    }
                    ew8(sb, db, i + 1);
                }
                tmem_st_wait();
            }
            fence_proxy_async_smem();   // dS^T (generic-proxy stores) -> visible to the tensor core
            tcgen05_fence_before();
            mbar_arrive(bar(EW_DONE0 + wg));
            if (stamp) bp.dbg[g * 8 + 2] = clock64();
            if (qb == nqb - 1) {
                // ---- last unit of the key tile: drain dV_kt and dK_kt (lane = key) ----
                const bool valid = inwin && j < S;
                const bool wload = __any_sync(0xffffffffu, valid);
                mbar_wait(bar(ACC_FULL), (li * nkt + kt) & 1);
                tcgen05_fence_after();
                bf16* dst = dbase + static_cast<long long>(j) * ld3;
                drain64(tm_acc, dst + 2 * p.H, 1.f, valid, wload);            // dV: P_drop already carries 1/(1-p)
                drain64(tm_acc + kHd, dst + p.H, p.scale, valid, wload);      // dK * 1/sqrt(d)
                tcgen05_fence_before();
                mbar_arrive(bar(ACC_EMPTY));
            }
            if (ul == upi - 1) {
                // ---- last unit of the item: drain dQ (lane = query), tile 0 then tile 1 ----
                mbar_wait(bar(DQ_FULL), li & 1);
                tcgen05_fence_after();
                for (int m = 0; m < (npq > kRows ? 2 : 1); ++m) {
                    const int q = m * kRows + r;
                    const bool valid = q < S;
                    const bool wload = __any_sync(0xffffffffu, valid);
                    drain64(tm_dq + m * kHd, dbase + static_cast<long long>(q) * ld3, p.scale, valid, wload);
                }
                tcgen05_fence_before();
                mbar_arrive(bar(DQ_EMPTY));
            }
            if (stamp) bp.dbg[g * 8 + 3] = clock64();
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 2) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

}  // namespace

static bool bwd_tc_config(const AttnParams& p, BwParams& bp) {
    if (p.S < 1 || p.S > kMaxNpq || (p.H % 8) != 0) return false;
    bp.a = p;
    bp.npq = (p.S + 15) / 16 * 16;
    bp.nqb = (bp.npq + 63) / 64;
    bp.nkt = p.S > kRows ? 2 : 1;
    bp.r2 = bp.nkt == 2 ? p.S - kRows : 0;
    bp.r2pad = (bp.r2 + 15) / 16 * 16;
    bp.nkb = (p.S + kBlk - 1) / kBlk;
    bp.nstage = bw_layout(bp.npq, bp.r2pad, 2).total <= 227 * 1024 ? 2 : 1;
    return bw_layout(bp.npq, bp.r2pad, bp.nstage).total <= 227 * 1024;
}

bool attn_bwd_tc_supported(const AttnParams& p) {
    BwParams bp;
    return bwd_tc_config(p, bp) && (reinterpret_cast<uintptr_t>(p.qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.dctx) & 15) == 0 &&
           (reinterpret_cast<uintptr_t>(p.dqkv) & 31) == 0;
}

// dQ | dK | dV of one layer call; p.drow must already hold D = rowsum(dO * O) (attn_delta_kernel)
int attn_bwd_tc(const AttnParams& p, cudaStream_t st) {
    BwParams bp;
    VB_REQUIRE(bwd_tc_config(p, bp), "attention backward (tcgen05): unsupported shape S=%d", p.S);
    const BwLayout L = bw_layout(bp.npq, bp.r2pad, bp.nstage);
    CUtensorMap tq, tdo, tk0, tk1;
    int rc = make_tmap_3d(&tq, p.qkv, p.S, p.B, 3 * p.H, bp.npq);
    if (rc) return rc;
    rc = make_tmap_3d(&tdo, p.dctx, p.S, p.B, p.H, bp.npq);
    if (rc) return rc;
    rc = make_tmap_3d(&tk0, p.qkv, p.S, p.B, 3 * p.H, kRows);
    if (rc) return rc;
    rc = make_tmap_3d(&tk1, p.qkv, p.S, p.B, 3 * p.H, bp.nkt == 2 ? bp.r2pad : 16);
    if (rc) return rc;
    static int configured[kMaxDevices] = {0};
    VB_CHECK_CUDA(ensure_dyn_smem(attn_bwd_tc_kernel, L.total, configured));
    const int total = p.B * p.A;
    const int grid = total < num_sms() ? total : num_sms();
    static long long* dbg_buf = nullptr;
    static int dbg_calls = 0;
    const char* de = getenv("VB_TC_DEBUG");
    bp.dbg = nullptr;
    if (de != nullptr && atoi(de) != 0) {
        if (dbg_buf == nullptr) cudaMallocManaged(&dbg_buf, 48 * 8 * sizeof(long long));
        bp.dbg = dbg_buf;
    }
    {
        ProfScope ps(st, PROF_ATTN_DKV, 8.0 * p.B * p.A * p.S * p.S * kHd, 1);
        VB_CHECK_CUDA(launch_pdl(attn_bwd_tc_kernel, dim3(grid), dim3(kThreadsBw), static_cast<size_t>(L.total), st, tq, tdo, tk0, tk1, bp));
    }
    VB_CHECK_CUDA(cudaGetLastError());
    if (bp.dbg != nullptr && ++dbg_calls == 3) {
        cudaStreamSynchronize(st);
        const long long t0 = dbg_buf[0];
        printf("tc attention backward timeline (CTA 0, cycles; unit g -> warp-group g %% 2)\n"
               " unit: ew_start sd_ready ew_done unit_end | mma: wait_ew ew_done_seen mmas_issued sd_issued(for this unit)\n");
        for (int i = 12; i < 36; ++i) {
            const long long* t = dbg_buf + i * 8;
            printf("  %2d: %7lld %7lld %7lld %7lld | %7lld %7lld %7lld %7lld\n", i, t[0] - t0, t[1] - t0, t[2] - t0, t[3] - t0, t[4] - t0,
                   t[5] - t0, t[6] - t0, t[7] - t0);
        }
    }
    return 0;
}

}  // namespace vb
