// sp_kernel_r64.cuh — the N = 4096 "64 x 64" render kernel: the headline size, and the second stage of
// the four-step path for N = 8192..65536.
//
// Design note: ncu on the round-1 16 x 16 x 16 kernel (profiles/r01_ncu_summary_s4a_dbx.txt, since deleted)
// showed the L1/shared-memory data pipe as the binding unit (22.5 wavefronts per 32 samples: two
// exchanges = 8, two histogram atomics = 3.6, window + twiddle tables = 2.5, scattered 32-byte row
// stores = 4.3, ...).  This kernel is built around that number:
//   * 4096 = 64 x 64: a thread holds 64 complex points, a frame is transformed by 64 threads with
//     ONE shared-memory exchange (4 wavefronts per 32 samples instead of 8), read back with LDS.128;
//   * ONE histogram atomic per pixel: the dB bin r and the colour index g are both monotone in
//     log2|X|^2, so the joint index r + (cmax - g) determines the pair; it is formed by FFMA.SAT +
//     FFMA on a 2^23 "magic" bias (no F2I, no integer clamps) and decoded once per render by
//     finalize_kernel (jh_decode);
//   * colour indices are staged as bytes in shared memory (two halves of 8 consecutive frames), so the
//     transposed image store (lib/worker.js:117) writes one full 32-byte sector per row and needs no
//     registers; the LUT + store work of a finished half is done by a third warpgroup of four STORE
//     warps (full / empty mbarriers, no CTA-wide barrier; register budget moved to the FFT warps with
//     setmaxnreg), so it runs beside the FFT arithmetic instead of inside its instruction stream;
//   * four independent frame streams per CTA (64 threads = 2 warps each, named barriers), one
//     persistent CTA per SM; the raw bytes of a stream's next frame are prefetched by one TMA bulk
//     copy INTO the stream's exchange buffer while the current frame is in registers.
// Only full tiles of frames that lie inside the buffer come here (spectrogram layout, cmap_len <= 256);
// the engine routes everything else through render_kernel.
// Replaces the hot loops of reference lib/worker.js:68-137 (+ lib/samples.js:313-400,
// lib/fft_nayuki.js:54-96).
#pragma once
#include "sp_fused.cuh"

namespace sp {

template <int FMT, bool SUB> struct R64Cfg {
    static constexpr int N = 4096, T = 64, STREAMS = 4, FFT_THREADS = T * STREAMS, STORE_THREADS = 128, THREADS = FFT_THREADS + STORE_THREADS;
    static constexpr int STEPS = 4, F = STREAMS * STEPS;                         // 16 frames per tile
    static constexpr int FFT_REGS = 232, STORE_REGS = 40;                        // 256 * 232 + 128 * 40 == 384 * 168, the CTA's allocation at launch: setmaxnreg only moves registers inside it
    static constexpr int SWB = SUB ? 8 : sample_width(FMT == FMT_RUNTIME ? CF64 : FMT);
    static constexpr bool OK = SUB || ((FMT != FMT_RUNTIME) && SWB <= 8);       // raw frame fits the exchange buffer
    static constexpr int XP = 66;                                                // exchange row pitch (float2): LDS.128 conflict-free
    static constexpr int X_BYTES = 64 * XP * 8;                                  // 33 792 >= 4096 * 8 + 32
    static constexpr int TW_PITCH = 14;                                          // float2 per thread row: w^1..w^7, w^8, w^16 .. w^56
    static constexpr int ST_PITCH = 1026;                                        // staging words per frame (1024 used)
    static constexpr int RING = 4;                                               // tile indices handed from the store warps' ticket thread to the CTA
    // the store warps' RGBA tiles (one 4 KB tile per warp: four boxes of 32 rows x 8 frames) for the tensor-TMA row stores; the
    // window comes from global memory (p.window_t, 16 KB: it stays in the 28 KB of L1 that the shared-memory carve-out leaves,
    // because nothing else of this kernel goes through L1)
    static constexpr int TILE_BYTES = (STORE_THREADS / 32) * 4096;
    static constexpr size_t SMEM_BYTES = (size_t)STREAMS * X_BYTES + (size_t)F * ST_PITCH * 4 + (size_t)JH_SIZE * 4
                                       + TILE_BYTES + (size_t)T * TW_PITCH * 8 + 1024 /* LUT */
                                       + (size_t)F * 2 * 8 /* s_mm */ + (size_t)2 * F * 8 /* s_fmid */ + 192 + 1024 /* LUT alignment */;
    static_assert(SMEM_BYTES <= 232448, "render_r64_kernel: dynamic shared memory above the 227 KB an sm_100 CTA may have");
};

// tw14: [64][14] float2 = W_4096^{t*k}, k = 1..7, 8, 16, 24, 32, 40, 48, 56
// OPT = false: the plain spectrogram kernel (the headline path, nothing else compiled in); OPT = true: the same kernel with
// the waterfall rows and the split-real post-process compiled in (selected by the launcher when a message asks for them),
// so that the options cost the plain kernel neither registers nor instruction-cache footprint.
template <int FMT, bool SUB, bool OPT = false>
__global__ void __launch_bounds__(384, 1) render_r64_kernel(const Params p, const float2 *__restrict__ tw14, const __grid_constant__ CUtensorMap tmap)
{
    using B = R64Cfg<FMT, SUB>;
    constexpr int N = B::N, T = B::T, F = B::F;
    constexpr bool FLOAT_IN = SUB || FMT == CF32 || FMT == CF64 || FMT == FMT_RUNTIME;   // |X|^2 may be +inf / NaN
    extern __shared__ __align__(128) unsigned char smem_r64[];
    // the reversed RGBA LUT sits on a 1 KB boundary of the shared window so that a pixel's table address is
    // ((word >> shift) & 0x3fc) | lut_base: one SHF + one 3-input LOP3 per lookup
    const unsigned lut_base = (smem_u32(smem_r64) + 1023u) & ~1023u;
    unsigned char *s_x = smem_r64 + (lut_base - smem_u32(smem_r64)) + 1024;           // [4][X_BYTES] exchange / raw frame
    unsigned *s_lut = reinterpret_cast<unsigned *>(s_x - 1024);                       // [256] RGBA indexed by the staged byte (cmax - g, or g when range < 0)
    unsigned char *s_tiles = s_x + B::STREAMS * B::X_BYTES;                          // [4 store warps][4 boxes][32 rows][32 B] RGBA, 1 KB aligned
    unsigned *s_stage = reinterpret_cast<unsigned *>(s_tiles + B::TILE_BYTES);       // [16][1026] colour bytes (4 bins per word)
    unsigned *s_jh = s_stage + F * B::ST_PITCH;                                       // [JH_SIZE] joint histogram
    float2 *s_tw = reinterpret_cast<float2 *>(s_jh + JH_SIZE);                       // [64][14]
    uint2 *s_mm = reinterpret_cast<uint2 *>(s_tw + T * B::TW_PITCH);                  // [16][2] per-warp min/max bit patterns of |X|^2
    float2 *s_fmid = reinterpret_cast<float2 *>(s_mm + F * 2);                       // [2 tile parities][16] raw mid sample of each frame
    uint64_t *s_mbar = reinterpret_cast<uint64_t *>(s_fmid + 2 * F);                  // [4]
    int *s_off = reinterpret_cast<int *>(s_mbar + B::STREAMS);                        // [4][2] misalignment of the staged frame
    uint64_t *s_full = reinterpret_cast<uint64_t *>(s_off + B::STREAMS * 2);          // [2] staging half h holds 8 finished frames
    uint64_t *s_empty = s_full + 2;                                                   // [2] staging half h has been stored
    uint64_t *s_tready = s_empty + 2;                                                 // [RING] ring slot holds its next tile index
    long long *s_ring = reinterpret_cast<long long *>(s_tready + B::RING);            // [RING] tile j >= 1 of this CTA in slot (j - 1) % RING
    long long *s_tile0 = s_ring + B::RING;                                            // this CTA's first tile

    const int tid = threadIdx.x;
    const int s = tid >> 6;                 // stream
    const int t = tid & 63;
    float2 *X = reinterpret_cast<float2 *>(s_x + (size_t)s * B::X_BYTES);
    unsigned char *raw = reinterpret_cast<unsigned char *>(X);
    uint64_t *mbar = s_mbar + s;

    const JhConst jc = fused_prologue(p, s_jh, s_lut, tid, B::THREADS);
    for (int i = tid; i < T * B::TW_PITCH; i += B::THREADS) s_tw[i] = tw14[i];
    const unsigned jh_base = smem_u32(s_jh) - (JH_MAGIC_BITS << 2);      // address of joint bin j = S.bits * 4 + jh_base (mod 2^32)
    const int nfull = p.n_full, sub_r = p.sub_r;

    // t == 0 of a stream: start the bulk copy of chunk-relative frame xr (sub-sequence k0sub) into the stream's buffer
    auto stage = [&](long long xr, int k0sub, unsigned par) {
        if (xr >= p.chunk_frames) xr = p.chunk_frames - 1;              // frames past the end of a partial tile redo the last one
        const void *src;
        unsigned bytes;
        if constexpr (SUB) {
            src = p.sub_in + ((size_t)xr * sub_r + (size_t)k0sub) * N;
            bytes = N * 8;
            s_off[s * 2 + par] = 0;
        } else {
            const long long xgl = p.frame_first + p.chunk_first + xr;
            const long long p0 = (long long)__dadd_rn(0.5, __dmul_rn(p.stride, (double)xgl)) - p.sample_base;   // lib/worker.js:72
            const unsigned long long off = (unsigned long long)p0 * B::SWB, a0 = off & ~15ull;
            src = p.buf + a0;
            bytes = (unsigned)(((off - a0) + (unsigned long long)N * B::SWB + 15) & ~15ull);
            s_off[s * 2 + par] = (int)(off - a0);
        }
        tma_load_1d(raw, src, bytes, mbar);
    };
    // tile -> first chunk-relative frame, sub-sequence
    auto tile_xr0 = [&](long long tile) -> long long { return (SUB ? tile / sub_r : tile) * F; };

    // Tiles are taken from the launch's counter in the order CTAs ask for them, so that a CTA which starts early (programmatic
    // dependent launch: on an SM the previous render has left) or runs fast takes more of them.  Tickets ntiles .. ntiles + grid - 1
    // mean "no more tiles", one per CTA; the CTA that draws the last of them resets the counter.  The engine alternates two
    // counters by launch: the launch after next reuses this one, and it starts only once this launch has completed (see
    // griddep_launch_dependents below).  One thread of the store warps draws the tickets, one tile ahead, and publishes them
    // through the ring.  A slot is rewritten RING tiles later; by then the full / empty hand-off has taken every warp at least
    // two tiles past reading it (RING >= 3).
    auto ticket = [&]() -> long long {
        const unsigned long long k = atomicAdd(p.tile_ctr, 1ull);
        if (k == (unsigned long long)p.ntiles + gridDim.x - 1) atomicExch(p.tile_ctr, 0ull);
        return (long long)k;
    };
    auto ring_put = [&](unsigned j, long long tl) {
        s_ring[(j - 1) % B::RING] = tl;
        mbar_arrive(s_tready + (j - 1) % B::RING);
    };
    auto ring_get = [&](unsigned j) -> long long {
        mbar_wait(s_tready + (j - 1) % B::RING, ((j - 1) / B::RING) & 1);
        return s_ring[(j - 1) % B::RING];
    };

    if (p.t_stamp && blockIdx.x == 0 && tid == 0) p.t_stamp[0] = globaltimer_ns();   // engine-owned: read only after the stream has drained
    if (t == 0 && tid < B::FFT_THREADS) mbar_init(mbar, 1);
    if (tid == 0) {
        for (int h = 0; h < 2; h++) { mbar_init(s_full + h, B::FFT_THREADS / 32); mbar_init(s_empty + h, B::STORE_THREADS / 32); }
        for (int r = 0; r < B::RING; r++) mbar_init(s_tready + r, 1);
    }
    if (tid == B::FFT_THREADS) *s_tile0 = ticket();
    if (t == 0) asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    long long tile = *s_tile0;
    unsigned kk = 0;                        // tiles done by this CTA (phase of the full / empty barriers, ring position)

    if (tid >= B::FFT_THREADS) {
        // ================= store warps: staged colour bytes -> LUT -> image rows (lib/worker.js:115-121) =================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(B::STORE_REGS));
        const int ht = tid - B::FFT_THREADS;
        const bool rows_aligned = (p.nframes % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.image) & 31) == 0);
        if (ht == 0 && tile < p.ntiles) ring_put(1, ticket());
        // Everything before this point reads only the capture and constant tables and writes only shared memory (the FFT warps
        // never write global memory before the joint-histogram flush): every global write of the CTA comes after the wait.  The
        // trigger comes after it on every path, tiles or none, so "render i + 2 has started" implies that render i and the
        // finalize_kernel behind it have completed - which the tile counters and the engine's accumulators rely on.
        griddep_wait();
        griddep_launch_dependents();
        while (tile < p.ntiles) {
            const int k0sub = SUB ? (int)(tile % sub_r) : 0;
            const long long xr0 = tile_xr0(tile);
#pragma unroll 1
            for (int h = 0; h < 2; h++) {
                mbar_wait(s_full + h, kk & 1);
                const size_t x0 = (size_t)(p.chunk_first + xr0) + 8 * h;
                const bool live = xr0 + 8 * h < p.chunk_frames;        // partial last tile: chunk_frames is a multiple of 8
                if constexpr (OPT && !SUB) {
                    if (p.waterfall && live) {
                        // waterfall layout (lib/worker.js:116): frame x is image row nframes - 1 - x, bin b is column
                        // n - 1 - y = (b + n/2 - 1) mod n.  A staged word holds bins k0 + 64*(4m + j): for a fixed (m, j) the
                        // lanes' bins - and columns - are consecutive, so every store instruction writes 128 contiguous bytes.
#pragma unroll 1
                        for (int f = 0; f < 8; f++) {
                            uint32_t *rowp = reinterpret_cast<uint32_t *>(p.image) + (size_t)N * (size_t)(p.nframes - 1 - (long long)(x0 + f));
                            const unsigned *src = s_stage + (8 * h + f) * B::ST_PITCH + ht;
#pragma unroll
                            for (int i = 0; i < 8; i++) {
                                const int id = ht + B::STORE_THREADS * i, k0 = id & 63, m = id >> 6;
                                const unsigned w = src[B::STORE_THREADS * i];
#pragma unroll
                                for (int j = 0; j < 4; j++)
                                    rowp[(k0 + 64 * (4 * m + j) + N / 2 - 1) & (N - 1)] = lut_at(lut_base, w, j);
                            }
                        }
                    }
                }
                if constexpr (!SUB) {
                    if (p.use_tma && live && (!OPT || !p.waterfall)) {
                        // RGBA tiles + tensor-TMA stores.  In iteration i this warp holds bins kb .. kb + 31 (kb = 32*(w & 1) + 64*(4m + j))
                        // for j = 0..3: four boxes of 32 consecutive image rows y0 .. y0 + 31, y0 = (n/2 - kb - 31) mod n (row r of a
                        // box is bin kb + 31 - r), each row 8 frames = 32 bytes.  The tile uses the 32-byte TMA swizzle (16-byte chunk
                        // index ^= bit 2 of the row), which makes the STS.128 below bank-conflict free.  The one box that would wrap
                        // (kb = n/2: bin n/2 is row 0, its neighbours rows n-1, n-2, ...) is placed at y0 = n - 31, where row 31 falls
                        // outside the tensor and is clipped by the TMA unit; that row is written by its lane directly.
                        const int lane = ht & 31, wq = ht >> 5;
                        unsigned char *tile = s_tiles + wq * 4096;
                        const int r = 31 - lane;
                        const unsigned toff = (unsigned)(r * 32 + (((r >> 2) & 1) << 4));
#pragma unroll 1
                        for (int i = 0; i < 8; i++) {
                            const int id = ht + B::STORE_THREADS * i, k0 = id & 63, m = id >> 6;
                            const unsigned *src = s_stage + (8 * h) * B::ST_PITCH + m * 64 + k0;
                            unsigned w[8];
#pragma unroll
                            for (int f = 0; f < 8; f++) w[f] = src[f * B::ST_PITCH];
                            if (lane == 0) bulk_wait_read0();              // the previous iteration's boxes have left the tile
                            __syncwarp();
#pragma unroll
                            for (int j = 0; j < 4; j++) {
                                uint4 a, b;
                                lut_row8(lut_base, w, j, a, b);
                                *reinterpret_cast<uint4 *>(tile + j * 1024 + toff) = a;
                                *reinterpret_cast<uint4 *>(tile + j * 1024 + (toff ^ 16u)) = b;
                                if (k0 + 64 * (4 * m + j) == N / 2)        // bin n/2 -> image row 0
                                    st_global_256(reinterpret_cast<uint32_t *>(p.image) + x0, a, b);
                            }
                            fence_async_smem();
                            __syncwarp();
                            if (lane == 0) {
                                const int kb0 = (k0 & 32) + 256 * m;       // kb of j = 0
#pragma unroll
                                for (int j = 0; j < 4; j++)
                                    tma_store_2d(&tmap, smem_u32(tile + j * 1024), (int)x0, (N / 2 - (kb0 + 64 * j) - 31) & (N - 1));
                                bulk_commit();
                            }
                        }
                    }
                }
#pragma unroll 1
                for (int i = 0; i < ((live && (!OPT || SUB || !p.waterfall) && !(!SUB && p.use_tma)) ? 8 : 0); i++) {
                    // bins k0 + 64*(4m + j), j = 0..3, of the half's 8 frames: one 32-byte sector per row
                    const int id = ht + B::STORE_THREADS * i, k0 = id & 63, m = id >> 6;
                    const unsigned *src = s_stage + (8 * h) * B::ST_PITCH + m * 64 + k0;
                    unsigned w[8];
#pragma unroll
                    for (int f = 0; f < 8; f++) w[f] = src[f * B::ST_PITCH];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const int kb = k0 + 64 * (4 * m + j);
                        const int bin = SUB ? k0sub + sub_r * kb : kb;
                        const int y = (nfull / 2 - bin) & (nfull - 1);                         // lib/worker.js:90
                        uint32_t *rowp = reinterpret_cast<uint32_t *>(p.image) + (size_t)p.nframes * (size_t)y + x0;   // :117
                        uint4 a, b;
                        if (!(p.dbg & 4)) lut_row8(lut_base, w, j, a, b);
                        else { a = make_uint4(w[0], w[1], w[2], w[3]); b = make_uint4(w[4], w[5], w[6], w[7]); }
                        if (!(p.dbg & 1)) store_row8(rowp, a, b, rows_aligned);
                    }
                }
                if (ht < 8 && live) {
                    // per-frame min / max of the half's frames, folded across the two warps of their stream, as dB
                    const int fl = 8 * h + ht;
                    const long long xl = p.chunk_first + xr0 + fl;
                    const uint2 m0 = s_mm[fl * 2], m1 = s_mm[fl * 2 + 1];
                    const float2 db = frame_db(min(m0.x, m1.x), max(m0.y, m1.y), p);
                    if constexpr (SUB) {
                        atomicMin(reinterpret_cast<unsigned *>(p.fmin) + xl, f2ord(db.x));
                        atomicMax(reinterpret_cast<unsigned *>(p.fmax) + xl, f2ord(db.y));
                    } else { p.fmin[xl] = db.x; p.fmax[xl] = db.y; p.fmid[xl] = s_fmid[(kk & 1) * F + fl]; }
                }
                __syncwarp();                                   // this warp is done reading the half (and s_mm)
                if ((ht & 31) == 0) mbar_arrive(s_empty + h);
            }
            tile = ring_get(++kk);
            if (ht == 0 && tile < p.ntiles) ring_put(kk + 1, ticket());
        }
        if constexpr (!SUB) bulk_wait_read0();        // the tiles must outlive the last tensor stores
    } else {
    // ================= FFT warps: four frame streams =================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(B::FFT_REGS));
    unsigned fpar = 0;                      // parity of this stream's frame counter (mbarrier phase, s_off slot)
    if (t == 0 && tile < p.ntiles) stage(tile_xr0(tile) + s, SUB ? (int)(tile % sub_r) : 0, 0);

    while (tile < p.ntiles) {
        const int k0sub = SUB ? (int)(tile % sub_r) : 0;
        const long long xr0 = tile_xr0(tile);
        long long next_tile = 0;

#pragma unroll 1
        for (int step = 0; step < B::STEPS; step++) {
            const int fl = step * B::STREAMS + s;                       // frame of the tile handled by this stream now
            const bool valid = xr0 + fl < p.chunk_frames;               // false: past the end of a partial last tile (outputs suppressed)
            // chunk_frames is a multiple of 8, so the frames past the end are exactly staging half 1 of the last tile: nobody
            // reads that half, and their histogram atomics are pointed at it instead of being predicated pixel by pixel
            const unsigned jbase = valid ? jh_base : jh_base + (smem_u32(s_stage + 8 * B::ST_PITCH) - smem_u32(s_jh));
            int half = step >> 1;                                       // staging half of this frame
            // (opaque to the optimiser: with `step & 1` known, nvcc 12.9 folded 8*(step >> 1) into 4*step and
            // produced a misaligned mbarrier address)
            asm volatile("" : "+r"(half));
            if (step == B::STEPS - 1) next_tile = ring_get(kk + 1);      // published when the store warps began this tile
            cf v[64];
            const bool split = OPT && !SUB && p.channel_mode;           // split-real needs the buffer once more, see below
            auto prefetch = [&]() {
                if (step < B::STEPS - 1) stage(xr0 + fl + B::STREAMS, k0sub, fpar);
                else if (next_tile < p.ntiles) stage(tile_xr0(next_tile) + s, SUB ? (int)(next_tile % sub_r) : 0, fpar);
            };
            // ---------------- load + decode + window (lib/worker.js:70-75) ----------------
            // in the order the column transforms of pass A consume them (columns 0..3 need the even window quads, 4..7 the
            // odd ones), so that the first transforms start while the later loads are still in flight
            mbar_wait(mbar, fpar);
            if constexpr (SUB) {
#pragma unroll
                for (int n0 = 0; n0 < 8; n0++)
#pragma unroll
                    for (int n1 = 0; n1 < 8; n1++) v[8 * n1 + n0] = cld(reinterpret_cast<const float2 *>(raw) + T * (8 * n1 + n0) + t);
            } else {
                const unsigned char *rp = raw + s_off[s * 2 + fpar];
                const float4 *wrow = p.window_t + t;
#pragma unroll
                for (int qq = 0; qq < 16; qq++) {
                    const int q = 2 * (qq & 7) + (qq >> 3);
                    const float4 w = __ldg(wrow + 64 * q);
                    cf d[4];
#pragma unroll
                    for (int c = 0; c < 4; c++) d[c] = decode_raw_cf<FMT>(rp, T * (4 * q + c) + t, p.format);
                    // raw sample at p0 + n/2 (lib/worker.js:131-133); the power-of-two scale is exact.  The store warps write it out
                    // (no global writes here, see griddep_wait); by parity of the tile, as this runs before the wait for the half
                    if (q == 8 && t == 0 && valid) s_fmid[(kk & 1) * F + fl] = make_float2(cre(d[0]) * raw_scale<FMT>(), cim(d[0]) * raw_scale<FMT>());
                    v[4 * q] = cscale(d[0], w.x);     v[4 * q + 1] = cscale(d[1], w.y);
                    v[4 * q + 2] = cscale(d[2], w.z); v[4 * q + 3] = cscale(d[3], w.w);
                }
            }
            fpar ^= 1;
            // ---------------- pass A: DFT-64 over the slow input digit; the raw frame is released between its two stages ----------------
            dft64_between(v, [&] { stream_barrier(s); });
            // twiddles W^{t*k}, each product followed by its exchange store Z[k0][t]
            twiddle_store64(v, reinterpret_cast<const float4 *>(s_tw + t * B::TW_PITCH), [&](int k) { return X + k * B::XP + t; });
            stream_barrier(s);
            // ---------------- pass B: thread k0 = t, DFT-64 over b; v[k1] is bin t + 64*k1 ----------------
            {
                const float4 *row = reinterpret_cast<const float4 *>(X + t * B::XP);
#pragma unroll
                for (int mm = 0; mm < 32; mm++) {                       // columns (0, 1) first, then (2, 3), ...
                    const int m = 4 * (mm & 7) + (mm >> 3);
                    const float4 q = row[m];
                    v[2 * m] = cpk(q.x, q.y); v[2 * m + 1] = cpk(q.z, q.w);
                }
            }
            dft64_between(v, [&] {
                stream_barrier(s);                                      // the exchange buffer is free: prefetch the stream's next frame
                if (t == 0 && !split) prefetch();
            });
            // first frame of this stream in staging half step/2: the store warps must be done with the half (previous tile)
            if ((step & 1) == 0) mbar_wait(s_empty + half, (kk + 1) & 1);
            {
                {
                    if constexpr (OPT && !SUB) {
                        if (split) {
                            // ---------------- split-real post-process (lib/fft_nayuki.js:103-119) ----------------
                            // bin i = t + 64*k1 pairs with bin n - i = (64 - t) + 64*(63 - k1): thread 64 - t, register 63 - k1 (thread 0
                            // pairs with itself, register 64 - k1).  One more pass through the exchange buffer: rows written with
                            // STS.128, the partner's row read back reversed with LDS.128 (both conflict-free at this pitch).
                            auto split_lo = [](cf a, cf b) {                    // i < n/2:  (re_i + re_p, im_i - im_p) / 2
                                const float2 fb = cun(b);
                                return cscale(cadd(a, cpk(fb.x, -fb.y)), 0.5f);
                            };
                            auto split_hi = [](cf a, cf b) {                    // i > n/2:  (im_p + im_i, -re_p + re_i) / 2, p = n - i
                                const float2 fa = cun(a), fb = cun(b);
                                return cscale(cadd(cpk(fa.y, fa.x), cpk(fb.y, -fb.x)), 0.5f);
                            };
                            {
                                float4 *wrow = reinterpret_cast<float4 *>(X + t * B::XP);
#pragma unroll
                                for (int m = 0; m < 32; m++) {
                                    const float2 a = cun(v[2 * m]), b = cun(v[2 * m + 1]);
                                    wrow[m] = make_float4(a.x, a.y, b.x, b.y);
                                }
                            }
                            stream_barrier(s);
                            if (t == 0) {
#pragma unroll
                                for (int k1 = 1; k1 < 32; k1++) {
                                    const cf a = v[k1], b = v[64 - k1];
                                    v[k1] = split_lo(a, b);
                                    v[64 - k1] = split_hi(b, a);
                                }
                                v[0] = cpk(fmaf(0.0f, cim(v[0]), cre(v[0])), 0.0f);   // imag[0] = 0; a NaN there reaches real[0] in the reference (NaN * 0)
                                v[32] = cpk(0.0f, 0.0f);                        // real[n/2] = imag[0] (just zeroed), imag[n/2] = 0
                            } else {
                                const float4 *prow = reinterpret_cast<const float4 *>(X + (64 - t) * B::XP);
#pragma unroll
                                for (int a = 0; a < 32; a++) {
                                    const float4 q = prow[31 - a];              // partner registers 62 - 2a (.xy) and 63 - 2a (.zw)
                                    if (a < 16) {
                                        v[2 * a] = split_lo(v[2 * a], cpk(q.z, q.w));
                                        v[2 * a + 1] = split_lo(v[2 * a + 1], cpk(q.x, q.y));
                                    } else {
                                        v[2 * a] = split_hi(v[2 * a], cpk(q.z, q.w));
                                        v[2 * a + 1] = split_hi(v[2 * a + 1], cpk(q.x, q.y));
                                    }
                                }
                            }
                            stream_barrier(s);                                  // now the buffer is free
                            if (t == 0) prefetch();
                        }
                    }

                    // ---------------- per-bin epilogue (lib/worker.js:85-122) ----------------
                    BinMinMax<FLOAT_IN> bm;
                    unsigned *stg = s_stage + fl * B::ST_PITCH + t;
#pragma unroll
                    for (int m = 0; m < 16; m++)                        // bins t + 64*(4m .. 4m+3) of frame fl: four colour bytes in one word
                        stg[m * 64] = epilogue4(v + 4 * m, bm, jc, jbase, true, 0u);
                    unsigned umn = __reduce_min_sync(0xffffffffu, bm.lo()), umx = __reduce_max_sync(0xffffffffu, bm.hi());
                    if (umn < 0x00800000u || umx >= 0x7f800000u)        // rare (warp-uniform)
                        fixup_nonfinite(v, true, (t & 31) == 0, valid, s_jh, jc, WarpMin(), WarpMax(), umn, umx);
                    if ((t & 31) == 0) s_mm[fl * 2 + (t >> 5)] = make_uint2(umn, umx);
                    if (step & 1) {                 // this warp has staged its last frame of half step/2 (and its s_mm entries)
                        __syncwarp();
                        if ((t & 31) == 0) mbar_arrive(s_full + half);
                    }
                }
            }
        } // steps
        tile = next_tile;
        kk++;
    } // tiles
    } // FFT warps

    __syncthreads();
    griddep_wait();                         // (the FFT warps' first global write)
    flush_joint_hist(p, s_jh, tid, B::THREADS);
}

} // namespace sp
