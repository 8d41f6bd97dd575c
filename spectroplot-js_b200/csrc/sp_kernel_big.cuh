// sp_kernel_big.cuh — n = R * 4096 (R = 2 .. 64, n = 8192 .. 262144) in ONE persistent launch: the four-step FFT
// of lib/fft_nayuki.js:54-96 with its intermediate kept in an L2-resident ring instead of a round trip through HBM.
//
// Round 1 ran the radix-R pre-pass and the 4096-point second stage as two kernels over a 1 GB scratch: 8 B/sample
// written to HBM and 8 B/sample read back on top of the 12 algorithmic bytes (ncu: 2.33 x the algorithmic traffic, C5 at
// 26 % of the HBM roofline).  Here both stages are work items of one persistent kernel (one CTA per SM) that walks an
// ordered queue:
//   P(b, jg)     pre-pass of points 256 jg .. 256 jg + 255 of the 8 frames of block b: decode + window + DFT_R over the slowest
//                input digit + twiddle W_n^{j k}, written as R sub-sequences of 4096 points per frame into ring slot b mod S;
//   F(b, i)      second stage of sub-sequences 2i and 2i + 1 of the 8 frames of block b: the 64 x 64 transform, dB, joint
//                histogram, colour bytes and image rows of render_r64_kernel, read from the ring with L2-only loads.
// Order: P of the first L blocks, then F(g) followed by P(g + L) for g = 0, 1, ...  An item waits only for items that
// come EARLIER in the queue (F(b) for the 16 P items of block b, P(b) for the F items of block b - S that used the slot
// before), every earlier item is held by a resident CTA that never waits for a later one, so the queue cannot deadlock;
// the hand-off is a release (stores, __threadfence, CTA barrier, atomicAdd) / acquire (ld.acquire, CTA barrier, ld.cg)
// pair per item.  The ring is S blocks = S * 8 * n * 8 bytes (32 MB for n = 65536 at S = 8), pinned in L2 by the engine
// (persisting access-policy window), so the pre-pass output never reaches HBM: DRAM traffic = input + image.
// Replaces the hot loops of reference lib/worker.js:68-137 (+ lib/samples.js:313-400, lib/fft_nayuki.js:54-96) for n > 4096.
#pragma once
#include "sp_fused.cuh"

namespace sp {

struct BigArgs {
    float2 *ring;              // [S][8][R][4096] complex fp32 sub-sequences
    const float2 *twT;         // [R - 1][4096]: W_n^{j*k}, k = 1 .. R-1 (double -> fp32 once), j fastest: coalesced
    unsigned *ctl;             // [0] queue head, [1 .. S] P items finished per slot, [1 + S .. 2S] F items finished per slot (zeroed per launch)
    int slots, lead;           // S, L
    long long nblocks;         // blocks of 8 frames rendered by this launch (frames chunk_first .. chunk_first + 8*nblocks)
    int R;
    int dbg;                   // timing experiments (wrong output): 1 no ring stores, 2 no dft / twiddle in the pre-pass, 4 no fence
    unsigned long long *stats; // optional [8]: SM cycles summed over CTAs (thread 0's clock): P wait, P work, F wait, F work, P items, F items, idle tail
};

struct BigCfg {
    static constexpr int N = 4096, T = 64, STREAMS = 4, FFT_THREADS = 256, STORE_THREADS = 128, THREADS = 384;
    static constexpr int STEPS = 4, F = 16, FFT_REGS = 232, STORE_REGS = 40;
    static constexpr int XP = 66, X_BYTES = 64 * XP * 8, TW_PITCH = 14, ST_PITCH = 1026;
    static constexpr size_t SMEM_BYTES = (size_t)STREAMS * X_BYTES + (size_t)F * ST_PITCH * 4 + (size_t)JH_SIZE * 4 + (size_t)T * TW_PITCH * 8
                                       + 1024 /* LUT */ + (size_t)F * 2 * 8 + 256 + 1024 /* LUT alignment */;
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void fft_barrier() { asm volatile("bar.sync 6, 256;" ::: "memory"); }   // the eight FFT warps

// One pre-pass item: points j = 256*jg + tid of ALL 8 frames of a block.  A thread keeps its R window coefficients and its
// R - 1 twiddles W_n^{j k} in registers for the 8 frames (R <= 16), so the tables cost 1/8 of their bytes on the SM's L2 port
// (the pre-pass is bound there: 8 B/sample in, 8 B/sample out to the ring), and the loads of the next U frames are in flight
// while the current U are transformed and stored (two register buffers).
template <int R, int FMT>
__device__ __forceinline__ void big_prepass(const Params &p, const BigArgs &g, long long blk, int jg, float2 *slot, int tid)
{
    constexpr int U = R <= 8 ? 4 : (R == 16 ? 2 : 1);          // frames per register buffer
    constexpr bool CACHE = R <= 16, TWOBUF = R <= 32;
    const int j = jg * 256 + tid;
    const size_t frame_f2 = (size_t)R * 4096;
    float w[CACHE ? R : 1];
    float2 tw[CACHE ? R : 1];
    if constexpr (CACHE) {
#pragma unroll
        for (int a = 0; a < R; a++) w[a] = __ldg(p.window + 4096 * a + j);
#pragma unroll
        for (int k = 1; k < R; k++) tw[k] = __ldg(g.twT + (size_t)(k - 1) * 4096 + j);
    }
    auto load = [&](cf (&v)[U][R], int f0) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            const long long xgl = p.frame_first + p.chunk_first + blk * 8 + f0 + u;
            const long long p0 = (long long)__dadd_rn(0.5, __dmul_rn(p.stride, (double)xgl)) - p.sample_base;   // lib/worker.js:72
#pragma unroll
            for (int a = 0; a < R; a++) v[u][a] = decode_raw_cf<FMT>(p.buf, p0 + 4096 * a + j, p.format);
        }
    };
    auto finish = [&](cf (&v)[U][R], int f0) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            if (j == 0)       // sample p0 + n/2 (lib/worker.js:131)
                p.fmid[p.chunk_first + blk * 8 + f0 + u] = make_float2(cre(v[u][R / 2]) * raw_scale<FMT>(), cim(v[u][R / 2]) * raw_scale<FMT>());
#pragma unroll
            for (int a = 0; a < R; a++) v[u][a] = cscale(v[u][a], CACHE ? w[a] : __ldg(p.window + 4096 * a + j));
            dft<R>(v[u]);
#pragma unroll
            for (int k = 1; k < R; k++) v[u][k] = cmul(v[u][k], CACHE ? tw[k] : __ldg(g.twT + (size_t)(k - 1) * 4096 + j));
            float2 *dst = slot + (size_t)(f0 + u) * frame_f2 + j;
#pragma unroll
            for (int k = 0; k < R; k++) cst(dst + (size_t)k * 4096, v[u][k]);
        }
    };
    if constexpr (TWOBUF) {
        cf va[U][R], vb[U][R];
        load(va, 0);
#pragma unroll 1
        for (int f0 = 0; f0 < 8; f0 += 2 * U) {
            load(vb, f0 + U);
            finish(va, f0);
            if (f0 + 2 * U < 8) load(va, f0 + 2 * U);
            finish(vb, f0 + U);
        }
    } else {
        cf va[U][R];
#pragma unroll 1
        for (int f0 = 0; f0 < 8; f0 += U) { load(va, f0); finish(va, f0); }
    }
}

// The fast form of the item: PPT = 2 adjacent points per thread (items of 512 points x 8 frames), input staged by bulk TMA.
// What bounds the pre-pass is the SM's load / store issue rate, not HBM (measured: profiles/r02_big_kernel.txt - 8-byte
// per-thread loads, cp.async and stores cost 2 .. 8 issue cycles per warp instruction and a 256-point item needs 3 300 of
// them), so the raw bytes are brought in by the TMA unit (no LSU instruction at all: ONE thread issues R bulk copies of
// 512 samples per frame from a uniform loop - issued from the lanes of a warp they serialise on the uniform datapath), the
// ring is written with 128-bit stores, and the frame after next is in flight while the current one is transformed.
template <int R, int FMT> struct BigStage {
    static constexpr int SW = sample_width(FMT == FMT_RUNTIME ? CF64 : FMT);
    static constexpr int CAP = BigCfg::STREAMS * BigCfg::X_BYTES;
    static constexpr int PPT = 2 * R * (512 * SW + 32) <= CAP ? 2 : 1;           // points per thread
    static constexpr int PTS = 256 * PPT;                                      // points per item
    static constexpr int SEG = PTS * SW + 32;                                  // staged segment: 16 bytes of alignment slack at either end
    static constexpr bool OK = FMT != FMT_RUNTIME && 2 * R * (256 * SW + 32) <= CAP;
    static constexpr int NP = OK ? 4096 / PTS : 16;                            // items per block
};
template <int R, int FMT>
__device__ __forceinline__ void big_prepass_tma(const Params &p, const BigArgs &g, long long blk, int jg, float2 *slot, int tid,
                                                unsigned char *stage, uint64_t *bars, int *s_poff, unsigned &tpar)
{
    using C = BigStage<R, FMT>;
    constexpr int PPT = C::PPT, SEG = C::SEG, SW = C::SW;
    constexpr bool CACHE = R * PPT <= 32;                          // window + twiddles of the thread's points stay in registers for the 8 frames
    const int j = jg * C::PTS + tid * PPT;
    const size_t frame_f2 = (size_t)R * 4096;
    float w[CACHE ? R : 1][PPT];
    float2 tw[CACHE ? R : 1][PPT];
    // one thread: bulk copies of frame f (R segments of PTS samples) into buffer f & 1
    auto issue = [&](int f) {
        const int b = f & 1;
        const long long xgl = p.frame_first + p.chunk_first + blk * 8 + f;
        const long long p0 = (long long)__dadd_rn(0.5, __dmul_rn(p.stride, (double)xgl)) - p.sample_base;   // lib/worker.js:72
        const unsigned long long off = (unsigned long long)(p0 + jg * C::PTS) * SW;
        const unsigned bytes = (((unsigned)off & 15u) + (unsigned)C::PTS * SW + 15u) & ~15u;
        const unsigned char *src = p.buf + (off & ~15ull);
        const unsigned dst = smem_u32(stage) + (unsigned)b * (R * SEG), bar = smem_u32(bars + b);
        s_poff[b] = (int)(off & 15ull);
        fence_async_smem();                                        // the FFT warps' reads of this buffer (through the barrier) vs the async writes
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes * R) : "memory");
#pragma unroll
        for (int a = 0; a < R; a++)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(dst + a * SEG), "l"(src + (size_t)4096 * a * SW), "r"(bytes), "r"(bar) : "memory");
    };
    if (tid == 0) { issue(0); issue(1); }
    if constexpr (CACHE) {
#pragma unroll
        for (int a = 0; a < R; a++)
#pragma unroll
            for (int q = 0; q < PPT; q++) w[a][q] = __ldg(p.window + 4096 * a + j + q);
#pragma unroll
        for (int k = 1; k < R; k++)
#pragma unroll
            for (int q = 0; q < PPT; q++) tw[k][q] = __ldg(g.twT + (size_t)(k - 1) * 4096 + j + q);
    }
#pragma unroll 1
    for (int f = 0; f < 8; f++) {
        const int b = f & 1;
        fft_barrier();                                             // s_poff of this frame is visible
        mbar_wait(bars + b, (tpar >> b) & 1u);
        tpar ^= 1u << b;
        const unsigned char *fp = stage + b * (R * SEG) + s_poff[b];
        cf v[PPT][R];
#pragma unroll
        for (int a = 0; a < R; a++)
#pragma unroll
            for (int q = 0; q < PPT; q++) v[q][a] = decode_raw_cf<FMT>(fp + a * SEG, tid * PPT + q, p.format);
        fft_barrier();                                             // everyone has read buffer b: the frame after next may land in it
        if (tid == 0 && f + 2 < 8) issue(f + 2);
        if (j == 0)       // sample p0 + n/2 (lib/worker.js:131)
            p.fmid[p.chunk_first + blk * 8 + f] = make_float2(cre(v[0][R / 2]) * raw_scale<FMT>(), cim(v[0][R / 2]) * raw_scale<FMT>());
#pragma unroll
        for (int q = 0; q < PPT; q++) {
#pragma unroll
            for (int a = 0; a < R; a++) v[q][a] = cscale(v[q][a], CACHE ? w[a][q] : __ldg(p.window + 4096 * a + j + q));
            if (!(g.dbg & 2)) {
                dft<R>(v[q]);
#pragma unroll
                for (int k = 1; k < R; k++) v[q][k] = cmul(v[q][k], CACHE ? tw[k][q] : __ldg(g.twT + (size_t)(k - 1) * 4096 + j + q));
            }
        }
        float2 *dst = slot + (size_t)f * frame_f2 + j;
        if (!(g.dbg & 1)) {
#pragma unroll
            for (int k = 0; k < R; k++) {
                if constexpr (PPT == 2) {
                    const float2 x0 = cun(v[0][k]), x1 = cun(v[1][k]);
                    *reinterpret_cast<float4 *>(dst + (size_t)k * 4096) = make_float4(x0.x, x0.y, x1.x, x1.y);
                } else cst(dst + (size_t)k * 4096, v[0][k]);
            }
        } else if (cre(v[0][0]) == 1234.5f) cst(dst, v[0][1]);
    }
}
template <int R, int FMT>
__device__ __forceinline__ void big_prepass_any(const Params &p, const BigArgs &g, long long blk, int jg, float2 *slot, int tid,
                                                unsigned char *stage, uint64_t *bars, int *s_poff, unsigned &tpar)
{
    if constexpr (BigStage<R, FMT>::OK) big_prepass_tma<R, FMT>(p, g, blk, jg, slot, tid, stage, bars, s_poff, tpar);
    else big_prepass<R, FMT>(p, g, blk, jg, slot, tid);
}
template <int FMT> __host__ __device__ constexpr int big_items_per_block(int R)
{
    return R == 2 ? BigStage<2, FMT>::NP : R == 4 ? BigStage<4, FMT>::NP : R == 8 ? BigStage<8, FMT>::NP : R == 16 ? BigStage<16, FMT>::NP
         : R == 32 ? BigStage<32, FMT>::NP : BigStage<64, FMT>::NP;
}

// tw14: [64][14] float2 = W_4096^{t*k}, k = 1..7, 8, 16, .., 56
template <int FMT>
__global__ void __launch_bounds__(384, 1) render_big_kernel(const Params p, const BigArgs g, const float2 *__restrict__ tw14)
{
    using B = BigCfg;
    constexpr int T = B::T, F = B::F;
    extern __shared__ __align__(128) unsigned char smem_big[];
    const unsigned lut_base = (smem_u32(smem_big) + 1023u) & ~1023u;             // see render_r64_kernel
    unsigned char *s_x = smem_big + (lut_base - smem_u32(smem_big)) + 1024;      // [4][X_BYTES] exchange buffers
    unsigned *s_lut = reinterpret_cast<unsigned *>(s_x - 1024);                  // [256] RGBA indexed by the staged byte
    unsigned *s_stage = reinterpret_cast<unsigned *>(s_x + B::STREAMS * B::X_BYTES);   // [16][1026] colour bytes (4 bins per word)
    unsigned *s_jh = s_stage + F * B::ST_PITCH;                                  // [JH_SIZE] joint histogram
    float2 *s_tw = reinterpret_cast<float2 *>(s_jh + JH_SIZE);                   // [64][14]
    uint2 *s_mm = reinterpret_cast<uint2 *>(s_tw + T * B::TW_PITCH);             // [16][2] per-warp min/max bit patterns of |X|^2
    uint64_t *s_full = reinterpret_cast<uint64_t *>(s_mm + F * 2);               // [2] staging half h holds 8 finished frames
    uint64_t *s_empty = s_full + 2;                                              // [2] staging half h has been stored
    long long *s_desc = reinterpret_cast<long long *>(s_empty + 2);              // [2][2] per F tile: first frame (chunk relative; -1 = stop), first sub-sequence
    volatile unsigned *s_item = reinterpret_cast<volatile unsigned *>(s_desc + 4);   // [1] item handed to the FFT warps
    uint64_t *s_pbar = reinterpret_cast<uint64_t *>(s_desc + 5);                 // [2] pre-pass frame landed
    int *s_poff = reinterpret_cast<int *>(s_pbar + 2);                           // [2] misalignment of the staged frame

    const int tid = threadIdx.x;
    const int s = tid >> 6, t = tid & 63;
    float2 *X = reinterpret_cast<float2 *>(s_x + (size_t)s * B::X_BYTES);

    const JhConst jc = fused_prologue(p, s_jh, s_lut, tid, B::THREADS);
    for (int i = tid; i < T * B::TW_PITCH; i += B::THREADS) s_tw[i] = tw14[i];
    const unsigned jh_base = smem_u32(s_jh) - (JH_MAGIC_BITS << 2);
    const int nfull = p.n_full, R = g.R;
    if (tid == 0) {
        for (int h = 0; h < 2; h++) { mbar_init(s_full + h, B::FFT_THREADS / 32); mbar_init(s_empty + h, B::STORE_THREADS / 32); mbar_init(s_pbar + h, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    unsigned kk = 0;                        // F tiles done by this CTA (phase of the full / empty barriers)

    if (tid >= B::FFT_THREADS) {
        // ================= store warps: staged colour bytes -> LUT -> image rows (lib/worker.js:115-121) =================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(B::STORE_REGS));
        const int ht = tid - B::FFT_THREADS;
        const bool rows_aligned = (p.nframes % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.image) & 31) == 0);
        for (;; kk++) {
            bool stop = false;
#pragma unroll 1
            for (int h = 0; h < 2; h++) {
                mbar_wait(s_full + h, kk & 1);
                const long long xr0 = s_desc[(kk & 1) * 2];
                if (xr0 < 0) { stop = true; break; }
                const int k0sub = (int)s_desc[(kk & 1) * 2 + 1] + h;
                const size_t x0 = (size_t)(p.chunk_first + xr0);
#pragma unroll 1
                for (int i = 0; i < 8; i++) {
                    // bins k0 + 64*(4m + j), j = 0..3, of the 8 frames of sub-sequence k0sub: one 32-byte sector per row
                    const int id = ht + B::STORE_THREADS * i, k0 = id & 63, m = id >> 6;
                    const unsigned *src = s_stage + (8 * h) * B::ST_PITCH + m * 64 + k0;
                    unsigned w[8];
#pragma unroll
                    for (int f = 0; f < 8; f++) w[f] = src[f * B::ST_PITCH];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const int bin = k0sub + R * (k0 + 64 * (4 * m + j));
                        const int y = (nfull / 2 - bin) & (nfull - 1);                         // lib/worker.js:90
                        uint32_t *rowp = reinterpret_cast<uint32_t *>(p.image) + (size_t)p.nframes * (size_t)y + x0;   // :117
                        uint4 a, b;
                        lut_row8(lut_base, w, j, a, b);
                        store_row8(rowp, a, b, rows_aligned);
                    }
                }
                if (ht < 8) {
                    // per-frame min / max folded across the two warps of a stream and across sub-sequences, as dB
                    const int fl = 8 * h + ht;
                    const long long xl = p.chunk_first + xr0 + ht;
                    const uint2 m0 = s_mm[fl * 2], m1 = s_mm[fl * 2 + 1];
                    const float2 db = frame_db(min(m0.x, m1.x), max(m0.y, m1.y), p);
                    atomicMin(reinterpret_cast<unsigned *>(p.fmin) + xl, f2ord(db.x));
                    atomicMax(reinterpret_cast<unsigned *>(p.fmax) + xl, f2ord(db.y));
                }
                __syncwarp();                                   // this warp is done reading the half (and s_mm)
                if ((ht & 31) == 0) mbar_arrive(s_empty + h);
            }
            if (stop) break;
        }
    } else {
        // ================= FFT warps: queue items =================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(B::FFT_REGS));
        const int S = g.slots, L = g.lead;
        const unsigned NP = (unsigned)big_items_per_block<FMT>(R), NF = (unsigned)(R / 2), G = NP + NF;
        unsigned tpar = 0;                  // parities of the two pre-pass frame barriers
        const unsigned long long pre = (unsigned long long)(g.nblocks < L ? g.nblocks : L) * NP;
        const unsigned long long total = pre + (unsigned long long)g.nblocks * G;
        const size_t frame_f2 = (size_t)R * 4096, slot_f2 = 8 * frame_f2;
        unsigned *q_head = g.ctl, *p_cnt = g.ctl + 1, *f_cnt = g.ctl + 1 + S;

        for (;;) {
            if (tid == 0) *s_item = atomicAdd(q_head, 1u);
            fft_barrier();
            const unsigned long long item = *s_item;
            fft_barrier();                                      // everyone has read the item before thread 0 overwrites it
            if (item >= total) break;
            // ---- decode the item
            bool is_f;
            long long blk;
            unsigned sub;
            if (item < pre) { is_f = false; blk = (long long)(item / NP); sub = (unsigned)(item % NP); }
            else {
                const unsigned long long i2 = item - pre;
                const long long grp = (long long)(i2 / G);
                const unsigned r = (unsigned)(i2 % G);
                if (r < NF) { is_f = true; blk = grp; sub = r; }
                else { is_f = false; blk = grp + L; sub = r - NF; }
            }
            if (blk >= g.nblocks) continue;                     // pre-pass slots past the last block
            const int slot = (int)(blk % S);
            const unsigned gen = (unsigned)(blk / S);
            float2 *ring = g.ring + (size_t)slot * slot_f2;

            long long c0 = 0, c1 = 0;
            if (g.stats && tid == 0) c0 = clock64();
            if (!is_f) {
                // ---------------- P: pre-pass of a quarter frame into the ring ----------------
                if (tid == 0) {
                    while (ld_acquire_u32(f_cnt + slot) < gen * NF) __nanosleep(200);             // the slot's previous block has been consumed
                    if (g.stats) c1 = clock64();
                }
                fft_barrier();
                switch (R) {
                case 2: big_prepass_any<2, FMT>(p, g, blk, (int)sub, ring, tid, s_x, s_pbar, s_poff, tpar); break;
                case 4: big_prepass_any<4, FMT>(p, g, blk, (int)sub, ring, tid, s_x, s_pbar, s_poff, tpar); break;
                case 8: big_prepass_any<8, FMT>(p, g, blk, (int)sub, ring, tid, s_x, s_pbar, s_poff, tpar); break;
                case 16: big_prepass_any<16, FMT>(p, g, blk, (int)sub, ring, tid, s_x, s_pbar, s_poff, tpar); break;
                case 32: big_prepass_any<32, FMT>(p, g, blk, (int)sub, ring, tid, s_x, s_pbar, s_poff, tpar); break;
                default: big_prepass_any<64, FMT>(p, g, blk, (int)sub, ring, tid, s_x, s_pbar, s_poff, tpar); break;
                }
                if (!(g.dbg & 4)) __threadfence();
                fft_barrier();
                if (tid == 0) {
                    atomicAdd(p_cnt + slot, 1u);
                    if (g.stats) { atomicAdd(g.stats + 0, (unsigned long long)(c1 - c0)); atomicAdd(g.stats + 1, (unsigned long long)(clock64() - c1)); atomicAdd(g.stats + 4, 1ull); }
                }
                continue;
            }

            // ---------------- F: sub-sequences 2*sub, 2*sub + 1 of the block's 8 frames ----------------
            if (tid == 0) {
                while (ld_acquire_u32(p_cnt + slot) < (gen + 1) * NP) __nanosleep(200);          // all 16 pre-pass items of the block have landed
                if (g.stats) c1 = clock64();
                s_desc[(kk & 1) * 2] = blk * 8;
                s_desc[(kk & 1) * 2 + 1] = 2 * sub;
            }
            fft_barrier();
#pragma unroll 1
            for (int step = 0; step < B::STEPS; step++) {
                const int fl = step * B::STREAMS + s;                       // slot of the tile handled by this stream now
                int half = step >> 1;                                       // staging half = sub-sequence of the pair
                asm volatile("" : "+r"(half));                              // (see render_r64_kernel)
                const float2 *src = ring + (size_t)(fl & 7) * frame_f2 + (size_t)(2 * sub + half) * 4096;
                cf v[64];
                // L2-only loads: the ring is rewritten by other SMs, an L1 line could be a generation old
#pragma unroll
                for (int a = 0; a < 64; a++) { const float2 q = __ldcg(src + T * a + t); v[a] = cpk(q.x, q.y); }

                // ---------------- pass A: DFT-64 over the slow input digit, twiddle W_4096^{t*k0} ----------------
                dft64_between(v, [&] { stream_barrier(s); });               // the previous frame's rows have been read back
                twiddle_store64(v, reinterpret_cast<const float4 *>(s_tw + t * B::TW_PITCH), [&](int k) { return X + k * B::XP + t; });
                stream_barrier(s);
                // ---------------- pass B: thread k0 = t, DFT-64 over b ----------------
                {
                    const float4 *row = reinterpret_cast<const float4 *>(X + t * B::XP);
#pragma unroll
                    for (int m = 0; m < 32; m++) {
                        const float4 q = row[m];
                        v[2 * m] = cpk(q.x, q.y); v[2 * m + 1] = cpk(q.z, q.w);
                    }
                }
                // first frame of this stream in staging half step/2: the store warps must be done with the half (previous tile)
                if ((step & 1) == 0) mbar_wait(s_empty + half, (kk + 1) & 1);
                dft<64>(v);                                                 // v[k1] is bin t + 64*k1 of the sub-sequence

                // ---------------- per-bin epilogue (lib/worker.js:85-122) ----------------
                BinMinMax<true> bm;
                unsigned *stg = s_stage + fl * B::ST_PITCH + t;
#pragma unroll
                for (int m = 0; m < 16; m++) stg[m * 64] = epilogue4(v + 4 * m, bm, jc, jh_base, true, 0u);
                unsigned umn = __reduce_min_sync(0xffffffffu, bm.lo()), umx = __reduce_max_sync(0xffffffffu, bm.hi());
                if (umn < 0x00800000u || umx >= 0x7f800000u)    // rare (warp-uniform)
                    fixup_nonfinite(v, true, (t & 31) == 0, true, s_jh, jc, WarpMin(), WarpMax(), umn, umx);
                if ((t & 31) == 0) s_mm[fl * 2 + (t >> 5)] = make_uint2(umn, umx);
                if (step & 1) {                 // this warp has staged its last frame of half step/2 (and its s_mm entries)
                    __syncwarp();
                    if ((t & 31) == 0) mbar_arrive(s_full + half);
                }
            } // steps
            kk++;
            // every ring read of this tile has been consumed (the loads of the last step were waited for by its pass A)
            fft_barrier();
            if (tid == 0) {
                __threadfence();
                atomicAdd(f_cnt + slot, 1u);
                if (g.stats) { atomicAdd(g.stats + 2, (unsigned long long)(c1 - c0)); atomicAdd(g.stats + 3, (unsigned long long)(clock64() - c1)); atomicAdd(g.stats + 5, 1ull); }
            }
        } // items

        // tell the store warps that no tile follows
        mbar_wait(s_empty + 0, (kk + 1) & 1);
        if (tid == 0) s_desc[(kk & 1) * 2] = -1;
        fft_barrier();
        if ((t & 31) == 0) mbar_arrive(s_full + 0);
    }

    __syncthreads();
    flush_joint_hist(p, s_jh, tid, B::THREADS);
}

} // namespace sp
