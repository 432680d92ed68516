// FAST-9/16 score map + cell-local strict 3x3 NMS + per-cell ini/min threshold selection, for every
// level of every image of the batch in ONE launch.
//
// Replaces the per-cell cv::FAST loop of ORBextractor::ComputeKeyPointsOctTree (reference
// src/ORBextractor.cc:784-829; OpenCV features2d/fast.cpp FAST_t<16> + cornerScore<16>) using the
// whole-level reformulation of SURVEY §8(a3), verified identical to the per-cell loop in
// tests/test_oracle_extract.py:
//   S(p)    = max over the 16 nine-pixel arcs (both polarities) of min |I_p - I_q|, minus 1
//             (p is a corner at threshold t  <=>  S(p) >= t);
//   keep(p) = S(p) strictly greater than S(q) for the 8-neighbours q that lie in the SAME cell's
//             detection domain (neighbours outside count as 0);
//   a cell emits keep(p) with S>=iniTh if any exists, else keep(p) with S>=minTh.
// One CTA owns `cellsPerBlk` whole cells of one cell row, so NMS and the threshold decision are CTA-local.
//
// Pipeline inside a CTA (v4):
//   0. one elected thread issues a 3-D TMA tile load (cp.async.bulk.tensor, box 160 x (hCell+6) bytes at
//      ((x0-4)&~15, y0-3, image): the inner start coordinate must be 16-byte aligned) into shared memory
//      and everybody waits on its mbarrier;
//   1a. a thread owns the 4 pixels of one ALIGNED 32-bit word of the tile and slides down its warp's rows with a
//      7-row register window.  Cheap reject: per even ring position one VABSDIFF4 gives |I_q - I_p| for the
//      4 pixels and three logic ops a per-byte ">t" flag; a FAST-9 arc contains a pixel of each antipodal
//      ring pair, so AND_j (f_j | f_{j+8}) == 0 rejects the pixel.  The surviving PIXELS (not words) go to the
//      warp's segment of a shared-memory pixel queue; ballots give their positions;
//   1b. each warp scores its queued pixels EXACTLY, two per thread in the two 16-bit lanes of a register, ring
//      bytes gathered with byte loads: S = max(max_k min_{j<9} I_{k+j} - I_p, I_p - min_k max_{j<9} I_{k+j}) - 1
//      with VIMNMX3.U16x2 (min3/max3) networks — the corner test IS the score (corner at t <=> S >= t).  The
//      corners are compacted in place to the front of the segment.  Pass A runs at iniThFAST only; cells that end
//      up without a kept corner are redone at minThFAST afterwards (pass B, same machinery), exactly the
//      reference's per-cell fallback;
//   2. cell-local strict NMS over each warp's corners, per-cell threshold decision and warp-aggregated append
//      to the global candidate list.
// Output: unordered candidate list per (image, level) of packed (x,y,score); consumers break ties with
// the reference's emission order key (cell row, cell col, y, x), never with list position.
//
// Bound (target): HBM read of the level pixels, once — sum_l w_l*h_l bytes per image.  Measured on B200: the
// integer ALU pipe (LOP3/PRMT/VABSDIFF4/VIMNMX3 all issue at 64 lanes/clk/SM, tools/ubench*.cu) — see DESIGN.md.
#include <cuda.h>

#include <cstring>

#include "borb_internal.h"

#include <algorithm>
#include <vector>

namespace borb {

namespace {

constexpr int TP = 160;                 // TMA box width == smem tile pitch (bytes).  TMA needs a 16-byte aligned start
                                        // column, so the box starts at xs = (x0-4) & ~15 and domain px xx sits at column xx+off
constexpr int TROWS = 66;               // hCell <= 60, + 3 halo rows above and below
constexpr int QCAP = 60 * 128;          // queue capacity >= every pixel of the largest tile

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 4-byte window starting DX bytes after the start of W1 (W0|W1|W2 are three consecutive aligned words)
template <int DX>
__device__ __forceinline__ uint32_t win(uint32_t W0, uint32_t W1, uint32_t W2) {
    if (DX == 0) return W1;
    if (DX > 0) return __byte_perm(W1, W2, DX | ((DX + 1) << 4) | ((DX + 2) << 8) | ((DX + 3) << 12));
    constexpr int K = 4 + DX;
    return __byte_perm(W0, W1, K | ((K + 1) << 4) | ((K + 2) << 8) | ((K + 3) << 12));
}

// CONSERVATIVE reject flag, 3 instructions (VABSDIFF4, IADD, LOP3): bit 7 of every byte of the result is set if that
// byte of a = |q - v| exceeds t (K = (127-t)*0x01010101, t <= 127).  Per byte a + (127-t) >= 128 <=> a > t; a byte whose
// sum overflows has a >= 129 (bit 7 of a itself, OR-ed in).  The carry out of an overflowing byte can raise the next
// byte's flag when that byte has a == t exactly: a false "keep", which only sends the word to the exact scoring pass
// (pass 1b decides every corner from exact scores), never a false reject.
__device__ __forceinline__ uint32_t gt_flag(uint32_t q, uint32_t v, uint32_t K) {
    const uint32_t a = __vabsdiffu4(q, v);
    return (a + K) | a;
}

// Two 16-bit lanes from two bytes held in the low byte of a and b: a in the low lane, b in the high lane.
__device__ __forceinline__ uint32_t pack2(uint32_t a, uint32_t b) { return __byte_perm(a, b, 0x5410); }

// Exact FAST scores of two pixels, one per 16-bit lane.  c0/c1 point at the pixels in the tile.  Returns S(p) clamped to
// [0,254] in each lane; S(p) >= t <=> p is a FAST-9 corner at threshold t (cornerScore<16> of OpenCV, both polarities at
// once).  min and max commute with subtracting I_p, so the arc networks run on the raw ring bytes and I_p is taken off at
// the end: bright = max_k min_{j<9} I_{k+j}, dark = min_k max_{j<9} I_{k+j}, S = max(bright - I_p, I_p - dark) - 1.
__device__ __forceinline__ uint32_t score_pair(const uint8_t* c0, const uint8_t* c1) {
    // Bresenham circle of radius 3, clockwise from (0,+3); only circular order matters
    constexpr int RX[16] = {0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1};
    constexpr int RY[16] = {3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3};
    uint32_t q[16];
#pragma unroll
    for (int k = 0; k < 16; k++) q[k] = pack2(c0[RY[k] * TP + RX[k]], c1[RY[k] * TP + RX[k]]);
    uint32_t lo3[16], hi3[16];
#pragma unroll
    for (int k = 0; k < 16; k++) {
        lo3[k] = __vimin3_u16x2(q[k], q[(k + 1) & 15], q[(k + 2) & 15]);
        hi3[k] = __vimax3_u16x2(q[k], q[(k + 1) & 15], q[(k + 2) & 15]);
    }
    uint32_t lo9[16], hi9[16];
#pragma unroll
    for (int k = 0; k < 16; k++) {
        lo9[k] = __vimin3_u16x2(lo3[k], lo3[(k + 3) & 15], lo3[(k + 6) & 15]);   // min over the arc k..k+8
        hi9[k] = __vimax3_u16x2(hi3[k], hi3[(k + 3) & 15], hi3[(k + 6) & 15]);   // max over the arc k..k+8
    }
    uint32_t bb[5], dd[5];
#pragma unroll
    for (int k = 0; k < 5; k++) {
        bb[k] = __vimax3_u16x2(lo9[3 * k], lo9[3 * k + 1], lo9[3 * k + 2]);
        dd[k] = __vimin3_u16x2(hi9[3 * k], hi9[3 * k + 1], hi9[3 * k + 2]);
    }
    const uint32_t bright = __vimax3_u16x2(__vimax3_u16x2(bb[0], bb[1], bb[2]), __vimax3_u16x2(bb[3], bb[4], lo9[15]), bb[0]);
    const uint32_t dark = __vimin3_u16x2(__vimin3_u16x2(dd[0], dd[1], dd[2]), __vimin3_u16x2(dd[3], dd[4], hi9[15]), dd[0]);
    const uint32_t v = pack2(c0[0], c1[0]);
    // lanes of bright - v and v - dark lie in [-255, 255]: S = max of the two - 1, clamped at 0
    return __viaddmax_s16x2_relu(__vmaxs2(__vsub2(bright, v), __vsub2(v, dark)), 0xFFFFFFFFu, 0u);
}

}  // namespace

struct TMaps { CUtensorMap m[BORB_MAX_LEVELS]; };

// One FAST CTA = whole cells of one cell row of one level.  The tile geometry is the same for every image of a batch, so it
// is computed once on the host (build_fast_tiles) instead of ~110 instructions per CTA (8.7 % of the kernel's instructions).
struct __align__(16) FastTile { int16_t l, ncell, x0, x1, y0, y1, wCell, hCell; };

__global__ void __launch_bounds__(256, 4) fast_kernel(const __grid_constant__ Geometry g, const __grid_constant__ TMaps tm,
                                                   const FastTile* __restrict__ tiles, uint32_t* __restrict__ cand, int* __restrict__ cand_cnt) {
    __shared__ __align__(128) uint8_t tile[TROWS * TP];
    __shared__ __align__(16) uint8_t score[60 * TP];     // S(p) in TILE coordinates (same columns as `tile`)
    // Pixel queue, entries = score-map offsets (row * TP + tile column).  Warp w owns the segment starting at yBeg * 128 (its
    // rows hold <= 128 domain pixels each), filled without atomics.  The dense pass compacts the segment's corners in place.
    __shared__ uint16_t pq[QCAP];
    __shared__ __align__(8) unsigned long long bar;
    __shared__ int needB;
    __shared__ int cellHasIni[128 / 30 + 1];
    __shared__ uint8_t cellOf[128];

    const int img = blockIdx.y;
    const FastTile T = tiles[blockIdx.x];                // one 16-byte load (only non-empty tiles are in the table)
    const int l = T.l, ncell = T.ncell, x0 = T.x0, x1 = T.x1, y0 = T.y0, y1 = T.y1;
    const int wCell = T.wCell, hCell = T.hCell;
    const LevelGeom& L = g.lv[l];
    const int tw = x1 - x0, th = y1 - y0;
    const int tid = threadIdx.x;
    const int lane = tid & 31, wrp = tid >> 5;
    const uint32_t ltmask = (1u << lane) - 1u;

    // ---- 0. TMA: tile rows y0-3 .. y0+hCell+2, columns xs .. xs+159 of image `img`, level l
    const int xs = (x0 - 4) & ~15;          // 16-byte aligned box start (TMA requirement)
    const int off = x0 - xs;                // tile column of domain pixel xx = 0   (4..19)
    if (tid == 0) {
        // the issuing thread initialises the barrier itself, so the copy starts before the CTA's first barrier; the other
        // threads see the initialised mbarrier after the __syncthreads() below and only then wait on it
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t bytes = (uint32_t)TP * (uint32_t)(hCell + 6);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&bar)), "r"(bytes) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
            ::"r"(smem_u32(tile)), "l"(reinterpret_cast<uint64_t>(&tm.m[l])), "r"(xs), "r"(y0 - 3), "r"(img), "r"(smem_u32(&bar))
            : "memory");
    }
    // overlap with the copy: bookkeeping
    if (tid < 128 / 30 + 1) cellHasIni[tid] = 0;
    if (tid < 128) cellOf[tid] = (uint8_t)(tid / wCell);
    if (tid == 0) needB = 0;
    __syncthreads();
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "FAST_TMA_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n"
        "@p bra FAST_TMA_DONE;\n"
        "bra FAST_TMA_WAIT;\n"
        "FAST_TMA_DONE:\n"
        "}\n" ::"r"(smem_u32(&bar))
        : "memory");
    // no CTA barrier here: every thread has observed the mbarrier phase itself (acquire), the bookkeeping stores above are
    // ordered by the __syncthreads() before the wait
    if (g.fast_mode == 1) {                 // ablation: tile load only (one word per thread consumed so the copy is observed)
        if (reinterpret_cast<const uint32_t*>(tile)[tid] == 0x12345678u && cand_cnt[0] == -1) cand[0] = 1;
        return;
    }

    const uint32_t* T32 = reinterpret_cast<const uint32_t*>(tile);
    uint32_t* S32 = reinterpret_cast<uint32_t*>(score);
    const int RG = (th + 7) >> 3;                 // rows per warp (8 warps)
    const int yBeg = wrp * RG, yEnd = min(th, yBeg + RG);
    uint16_t* seg = pq + yBeg * 128;
    const int wc = (off >> 2) + lane;             // lane owns aligned tile word wc (tile columns 4*wc .. 4*wc+3)
    uint32_t vmask = 0;                           // bit 7 of byte b: pixel 4*wc+b lies in the domain
#pragma unroll
    for (int b = 0; b < 4; b++)
        if (4 * wc + b - off >= 0 && 4 * wc + b - off < tw) vmask |= 0x80u << (8 * b);

    // Slides the warp down its rows yBeg..yEnd-1 with a rolling 7-row window of 3 words per lane.  Cheap reject at threshold t
    // (t <= 127; K = (127-t)*0x01010101): per even ring position one VABSDIFF4 gives |I_q - I_p| for the 4 pixels of the word
    // and gt_flag a per-byte ">t" flag; a FAST-9 arc contains a pixel of each antipodal ring pair, so a pixel whose
    // AND_j (f_j | f_{j+8}) is clear has S < t.  The surviving pixels among `mask` are appended to the warp's segment; ballots
    // place them, so no atomic is needed.  zero: also clear the score map of the domain words (rejected pixels read as 0).
    // Returns the number of queued pixels (warp-uniform).
    auto sweep = [&](uint32_t mask, int t, bool zero) -> int {
        const bool reject = t <= 127;
        const uint32_t K = (uint32_t)(127 - min(t, 127)) * 0x01010101u;
        uint32_t a0[7], a1[7], a2[7];
        int n = 0;
        if (yBeg < yEnd) {
#pragma unroll
            for (int j = 0; j < 6; j++) {
                const uint32_t* rp = T32 + (yBeg + j) * (TP / 4) + wc - 1;
                a0[j] = rp[0]; a1[j] = rp[1]; a2[j] = rp[2];
            }
        }
#pragma unroll
        for (int it = 0; it < 8; it++) {
            const int yy = yBeg + it;
            if (yy < yEnd) {          // warp-uniform
                {
                    const uint32_t* rp = T32 + (yy + 6) * (TP / 4) + wc - 1;
                    a0[(it + 6) % 7] = rp[0]; a1[(it + 6) % 7] = rp[1]; a2[(it + 6) % 7] = rp[2];
                }
#define ROW(dy) a0[(it + (dy) + 3) % 7], a1[(it + (dy) + 3) % 7], a2[(it + (dy) + 3) % 7]
                uint32_t m = mask;
                if (reject && m) {
                    const uint32_t v = a1[(it + 3) % 7];
                    uint32_t acc = gt_flag(win<0>(ROW(3)), v, K) | gt_flag(win<0>(ROW(-3)), v, K);      // pair (0,8)
                    acc &= gt_flag(win<2>(ROW(2)), v, K) | gt_flag(win<-2>(ROW(-2)), v, K);               // (2,10)
                    acc &= gt_flag(win<3>(ROW(0)), v, K) | gt_flag(win<-3>(ROW(0)), v, K);                // (4,12)
                    acc &= gt_flag(win<2>(ROW(-2)), v, K) | gt_flag(win<-2>(ROW(2)), v, K);               // (6,14)
                    m &= acc;
                }
#undef ROW
                if (zero && vmask) S32[yy * (TP / 4) + wc] = 0;
                const int e = yy * TP + 4 * wc;
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    const bool f = (m >> (8 * b + 7)) & 1u;
                    const unsigned bal = __ballot_sync(0xFFFFFFFFu, f);
                    if (f) seg[n + __popc(bal & ltmask)] = (uint16_t)(e + b);
                    n += __popc(bal);
                }
            }
        }
        return n;
    };

    // Exact scores of the warp's n queued pixels, two per lane (entries i and i+32 of each group of 64, so the lanes of one
    // load read consecutive queue entries: mostly distinct words of one row, few bank conflicts).  Writes S to the score map
    // and compacts the pixels with S >= max(t,1) to the front of the segment (writes never overtake reads); returns their count.
    auto dense = [&](int n, int t) -> int {
        const int tc = max(t, 1);
        int nc = 0;
        for (int b = 0; b < n; b += 64) {     // warp-uniform
            const int e0 = b + lane, e1 = e0 + 32;
            const int o0 = seg[min(e0, n - 1)], o1 = seg[min(e1, n - 1)];
            const uint32_t s = score_pair(tile + 3 * TP + o0, tile + 3 * TP + o1);   // tile row = score row + 3
            const int s0 = s & 0xFFFFu, s1 = s >> 16;
            const bool h0 = e0 < n, h1 = e1 < n;
            if (h0) score[o0] = (uint8_t)s0;
            if (h1) score[o1] = (uint8_t)s1;
            const bool c0 = h0 && s0 >= tc, c1 = h1 && s1 >= tc;
            const unsigned b0 = __ballot_sync(0xFFFFFFFFu, c0), b1 = __ballot_sync(0xFFFFFFFFu, c1);
            if (c0) seg[nc + __popc(b0 & ltmask)] = (uint16_t)o0;
            if (c1) seg[nc + __popc(b0) + __popc(b1 & ltmask)] = (uint16_t)o1;
            nc += __popc(b0) + __popc(b1);
        }
        __syncwarp();
        return nc;
    };

    // ---- 1. pass A at iniThFAST only: a cell falls back to minThFAST only if it has NO kept corner at iniThFAST
    //         (ORBextractor.cc:809-816), and a pixel with S < ini can neither be kept at ini nor suppress one that is.
    // No CTA barrier between the sweep and the dense pass: a warp zeroes, queues and scores only its own rows.
    const int nA = sweep(vmask, g.ini_th, true);
    if (g.fast_mode == 2) {                 // ablation: load + reject + pixel queue
        if (nA == -1) cand[0] = 1;
        return;
    }
    int nc = dense(nA, g.ini_th);
    __syncthreads();                        // the score map is complete
    if (g.fast_mode == 3) {                 // ablation: load + reject + exact scores
        if (nc == -1) cand[0] = 1;
        return;
    }

    uint32_t* out = cand + (size_t)img * g.cand_image_stride + L.cand_off;
    int* cnt = cand_cnt + img * g.nlevels + l;

    // cell-local strict NMS over the warp's corners seg[0..n) (0xFFFF = dropped), then a warp-aggregated append of the
    // survivors to the global candidate list; optionally records which cells keep something
    auto nms_emit = [&](int n, bool mark) {
        for (int eb = 0; eb < n; eb += 32) {  // warp-uniform
            const int e = eb + lane;
            int s = 0, xx = 0, yy = 0;
            if (e < n) {
                const int o = seg[e];
                yy = o / TP;
                const int col = o - yy * TP;
                xx = col - off;
                s = score[o];
                const int c = cellOf[xx];
                const int cx0 = c * wCell, cx1 = min(cx0 + wCell, tw);
                bool ismax = true;
#pragma unroll
                for (int dy = -1; dy <= 1; dy++)
#pragma unroll
                    for (int dx = -1; dx <= 1; dx++) {
                        if (dx == 0 && dy == 0) continue;
                        const int qx = xx + dx, qy = yy + dy;
                        if (qx < cx0 || qx >= cx1 || qy < 0 || qy >= th) continue;
                        if (!(s > (int)score[o + dy * TP + dx])) ismax = false;
                    }
                if (ismax) {
                    if (mark) cellHasIni[c] = 1;
                } else
                    s = 0;
            }
            const unsigned m = __ballot_sync(0xFFFFFFFFu, s > 0);
            if (m) {
                int base = 0;
                if (lane == 0) base = atomicAdd(cnt, __popc(m));
                base = __shfl_sync(0xFFFFFFFFu, base, 0);
                if (s > 0) {
                    const int pos = base + __popc(m & ltmask);
                    if (pos < L.cand_cap) out[pos] = pack_xys(x0 + xx, y0 + yy, s);
                }
            }
        }
    };

    // ---- 2. pass A: NMS among the S >= iniTh corners; every survivor is emitted and marks its cell
    nms_emit(nc, true);
    __syncthreads();
    if (tid < ncell && tid * wCell < tw && !cellHasIni[tid] && g.min_th < g.ini_th) needB = 1;
    __syncthreads();
    if (!needB) return;

    // ---- 3. pass B (rare): cells without any kept iniTh corner are redone at minThFAST (ORBextractor.cc:812-816).  Every
    //         pixel of those cells that passes the minTh reject is scored again, pass-A pixels included: a cell can hold
    //         iniTh corners and still keep none when strict NMS on a plateau suppresses them all, and then NMS at minTh
    //         needs the exact score of every pixel >= minTh.  Pixels the minTh reject drops have S < minTh; the score map
    //         holds 0 or their exact pass-A score for them, either of which NMS at minTh treats alike.
    {
        uint32_t need = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int xx = 4 * wc + b - off;
            if (xx >= 0 && xx < tw && !cellHasIni[cellOf[xx]]) need |= 0x80u << (8 * b);
        }
        if (__any_sync(0xFFFFFFFFu, need != 0)) {
            const int nB = sweep(need, g.min_th, false);
            nc = dense(nB, g.min_th);
        } else
            nc = 0;
        __syncthreads();                    // every pass-B score is in the score map
        nms_emit(nc, false);
    }
}

// ---- host: tensor maps (one per level: 3-D {x, y, image} view of the pyramid buffer)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

borb_status build_fast_tmaps(const Geometry& g, const Workspace& ws, void* out_tmaps) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
            set_error("cuTensorMapEncodeTiled unavailable (%s)", cudaGetErrorString(e));
            return BORB_ERR_CUDA;
        }
        encode = (EncodeTiledFn)fn;
    }
    TMaps* tm = reinterpret_cast<TMaps*>(out_tmaps);
    std::memset(tm, 0, sizeof(TMaps));
    for (int l = 0; l < g.nlevels; l++) {
        const LevelGeom& L = g.lv[l];
        cuuint64_t dims[3] = {(cuuint64_t)L.w, (cuuint64_t)L.h, (cuuint64_t)ws.max_images};
        cuuint64_t strides[2] = {(cuuint64_t)L.pitch, (cuuint64_t)g.pyr_image_stride};
        cuuint32_t box[3] = {(cuuint32_t)TP, (cuuint32_t)(L.hCell + 6), 1};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = encode(&tm->m[l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, ws.pyr + L.pyr_off, dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("cuTensorMapEncodeTiled failed for level %d (CUresult %d)", l, (int)r);
            return BORB_ERR_CUDA;
        }
    }
    return BORB_OK;
}

size_t fast_tmaps_bytes() { return sizeof(TMaps); }

// The non-empty tiles of one image in (level, cell row, block column) order - the order the grid had when the kernel derived
// the geometry itself (ORBextractor.cc:781-787 cell grid, cellsPerBlk cells per CTA).
borb_status build_fast_tiles(const Geometry& g, Workspace& ws) {
    std::vector<FastTile> t;
    for (int l = 0; l < g.nlevels; l++) {
        const LevelGeom& L = g.lv[l];
        for (int cellRow = 0; cellRow < L.nRows; cellRow++)
            for (int blkCol = 0; blkCol < L.blkCols; blkCol++) {
                const int cell0 = blkCol * L.cellsPerBlk;
                const int ncell = std::min(L.cellsPerBlk, L.nCols - cell0);
                const int x0 = EDGE + cell0 * L.wCell, x1 = std::min(x0 + ncell * L.wCell, L.w - EDGE);
                const int y0 = EDGE + cellRow * L.hCell, y1 = std::min(y0 + L.hCell, L.h - EDGE);
                if (x0 >= x1 || y0 >= y1) continue;
                FastTile f;
                f.l = (int16_t)l; f.ncell = (int16_t)ncell; f.x0 = (int16_t)x0; f.x1 = (int16_t)x1; f.y0 = (int16_t)y0; f.y1 = (int16_t)y1;
                f.wCell = (int16_t)L.wCell; f.hCell = (int16_t)L.hCell;
                t.push_back(f);
            }
    }
    cudaFree(ws.fast_tiles); ws.fast_tiles = nullptr;
    ws.fast_n_tiles = (int)t.size();
    if (t.empty()) return BORB_OK;
    BORB_CUDA(cudaMalloc(&ws.fast_tiles, t.size() * sizeof(FastTile)));
    BORB_CUDA(cudaMemcpy(ws.fast_tiles, t.data(), t.size() * sizeof(FastTile), cudaMemcpyHostToDevice));
    return BORB_OK;
}

int launch_fast(const Geometry& g, const Workspace& ws, int n_images, cudaStream_t s) {
    if (ws.fast_n_tiles == 0) return 0;
    dim3 grid(ws.fast_n_tiles, n_images);
    fast_kernel<<<grid, 256, 0, s>>>(g, *reinterpret_cast<const TMaps*>(ws.fast_tmaps), reinterpret_cast<const FastTile*>(ws.fast_tiles), ws.cand, ws.cand_cnt);
    return 1;
}

}  // namespace borb
