// Internal declarations of libborb (B200 / sm_100a ORB front-end).  Not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/borb.h"

namespace borb {

constexpr int EDGE = 19;          // EDGE_THRESHOLD   (ORBextractor.cc:74)
constexpr int PATCH = 31;         // PATCH_SIZE       (:72)
constexpr int HALF_PATCH = 15;    // HALF_PATCH_SIZE  (:73)
constexpr int MIN_BORDER = 16;    // EDGE_THRESHOLD-3 (:773)
constexpr int TH_HIGH = 100;      // ORBmatcher.cc:37
constexpr int TH_LOW = 50;        // ORBmatcher.cc:38
constexpr int BLUR_TILE_W = 120;  // blur strip: 30 output words per warp + one halo word each side
constexpr int BLUR_TILE_H = 64;   // rows per blur CTA
constexpr int FAST_TILE_W = 124;  // max detection-domain width of one FAST CTA (<= 32 aligned words incl. misalignment)

// Candidate / selected-keypoint record: x | y<<12 | score<<24   (x,y <= 4095, score <= 255)
__host__ __device__ inline uint32_t pack_xys(int x, int y, int s) { return (uint32_t)x | ((uint32_t)y << 12) | ((uint32_t)s << 24); }
__host__ __device__ inline int xys_x(uint32_t v) { return (int)(v & 0xFFFu); }
__host__ __device__ inline int xys_y(uint32_t v) { return (int)((v >> 12) & 0xFFFu); }
__host__ __device__ inline int xys_s(uint32_t v) { return (int)(v >> 24); }

struct LevelGeom {
    int w, h;               // level size, cvRound(orig * invScale) (ORBextractor.cc:1111-1112)
    int pitch;              // bytes per row in the pyramid buffers
    unsigned pyr_off;       // byte offset of this level inside one image's pyramid block
    // FAST cell grid (ORBextractor.cc:781-787)
    int nCols, nRows, wCell, hCell;
    int cellsPerBlk;        // cells per FAST CTA along x
    int blkCols;            // CTAs per cell row
    int blkBase;            // first CTA of this level inside one image's FAST grid
    unsigned cand_off;      // entry offset of this level's candidate list inside one image's block
    int cand_cap;
    int quota;              // mnFeaturesPerLevel[level]
    int nIni;               // quadtree roots (ORBextractor.cc:543)
    float hX;               // (:545)
    int node_cap;           // max list size + slack
    int sel_off;            // entry offset of this level's selected list inside one image's block
    float scale;            // mvScaleFactor[level]
    float inv_scale;        // mvInvScaleFactor[level]
    float patch_size;       // (float)(int)(PATCH_SIZE*scale)  (:837)
    unsigned xtab_off, ytab_off;   // resize tables ({ofs, c0, c1, 0} int16 quadruples), in entries
    unsigned xwin_off;             // windowed x table ({c0, c1, group base, PRMT selectors}), in entries; see k_pyramid.cu
    int x_windowed;                // 1: every group of 4 destination columns reads inside one aligned 12-byte source window
};

struct Geometry {
    int nlevels;
    int w, h;
    int ini_th, min_th;
    int fast_mode;              // 0: full kernel.  Ablation (borb_debug_set_fast_mode): 1 = TMA tile load only, 2 = + packed reject
                                // and pixel queue, 3 = + exact pixel scores (no NMS / emit)
    int fast_blocks;            // FAST CTAs per image (all levels)
    unsigned pyr_image_stride;  // bytes
    unsigned cand_image_stride; // entries
    int sel_image_stride;       // entries  (== keypoint capacity per image)
    int blur_tiles;             // blur CTAs per image (all levels)
    int blur_base[BORB_MAX_LEVELS + 1];
    int umax[16];
    LevelGeom lv[BORB_MAX_LEVELS];
};

// Per-batch device buffers of one handle
struct Workspace {
    int max_images = 0;
    uint8_t* pyr = nullptr;        // max_images * pyr_image_stride
    uint8_t* blur = nullptr;       // same layout, GaussianBlur'ed levels
    uint32_t* cand = nullptr;      // max_images * cand_image_stride
    int* cand_cnt = nullptr;       // max_images * nlevels
    int* pnode = nullptr;          // quadtree scratch, same shape as cand
    uint32_t* sel = nullptr;       // max_images * sel_image_stride
    int* sel_cnt = nullptr;        // max_images * nlevels
    borb_keypoint* kps = nullptr;  // max_images * sel_image_stride
    uint8_t* desc = nullptr;       // max_images * sel_image_stride * 32
    int* nkp = nullptr;            // max_images
    float* u_right = nullptr;      // max_images/2+1 pairs * sel_image_stride
    float* depth = nullptr;
    int* sad = nullptr;            // SAD distance per left keypoint (-1: none)
    int16_t* tabs = nullptr;       // resize tables
    int* pair_idx = nullptr;       // 2 * max_pairs (left,right image indices)
    int* st_bins = nullptr;        // stereo row-bin offsets, per pair
    void* st_recs = nullptr;       // stereo binned right-keypoint records, per pair
    uint8_t* stage = nullptr;      // tightly packed H2D landing buffer (grow-only)
    size_t stage_bytes = 0;
    void* fast_tmaps = nullptr;    // HOST: per-level CUtensorMap set for fast_kernel (passed by value at launch)
    void* fast_tiles = nullptr;    // DEVICE: one 16-byte descriptor per FAST CTA of an image (k_fast.cu: FastTile), n = fast_n_tiles
    int fast_n_tiles = 0;
};

void set_error(const char* fmt, ...);
// Raises `func`'s dynamic shared-memory limit to the device's opt-in maximum (minus the kernel's static shared memory),
// ONCE per (kernel, device) under a mutex.  The attribute is per function and per device and is shared by every handle
// on every host thread, so it must never be lowered between another thread's set and launch (handles on the Tracking,
// LocalMapping and LoopClosing threads launch the same kernels concurrently).  Returns false (and sets the error) on failure.
bool allow_max_smem(const void* func);
#define BORB_CUDA(call)                                                                             \
    do {                                                                                            \
        cudaError_t _e = (call);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            borb::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return (_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver) ? BORB_ERR_NO_DEVICE : BORB_ERR_CUDA; \
        }                                                                                           \
    } while (0)

// ---- kernel launchers (each returns the number of kernel launches it issued) -----------------
int launch_repack_remap(const Geometry& g, const Workspace& ws, const uint8_t* stage, int src_stride, size_t src_image_bytes, int src_w,
                        int src_h, const float* mx0, const float* my0, const float* mx1, const float* my1, int n_images, cudaStream_t s);
int launch_repack_color(const Geometry& g, const Workspace& ws, const uint8_t* stage, int src_stride, size_t src_image_bytes, int channels,
                        int rgb, int n_images, cudaStream_t s);
int launch_repack(const Geometry& g, const Workspace& ws, const uint8_t* stage, int src_stride, size_t src_image_bytes,
                  int n_images, cudaStream_t s);
int launch_pyramid(const Geometry& g, const Workspace& ws, int n_images, cudaStream_t s);
int launch_fast(const Geometry& g, const Workspace& ws, int n_images, cudaStream_t s);
int launch_quadtree(const Geometry& g, const Workspace& ws, int n_images, cudaStream_t s);
int launch_blur(const Geometry& g, const Workspace& ws, int n_images, cudaStream_t s);
int launch_describe(const Geometry& g, const Workspace& ws, int n_images, cudaStream_t s);

struct StereoView {          // device pointers of one side of a stereo pair set
    const uint8_t* pyr;      // pyramid base (image 0)
    const borb_keypoint* kps;
    const uint8_t* desc;
    const int* nkp;
    unsigned pyr_image_stride;
    int kp_image_stride;
};
int launch_stereo(const Geometry& g, const StereoView& L, const StereoView& R, const int* d_pair_idx, int n_pairs,
                  float bf, float b, float* d_u_right, float* d_depth, int* d_sad, int out_stride, int* d_bins, void* d_recs,
                  cudaStream_t s);
int stereo_rec_stride(const Geometry& g);
size_t stereo_bins_bytes_per_pair();
size_t stereo_rec_bytes();
size_t quadtree_smem_bytes(int node_cap);
borb_status build_fast_tmaps(const Geometry& g, const Workspace& ws, void* out_tmaps);
borb_status build_fast_tiles(const Geometry& g, Workspace& ws);
size_t fast_tmaps_bytes();

}  // namespace borb

struct borb_extractor {
    borb_extractor_cfg cfg;
    int device = 0;
    cudaStream_t stream = nullptr;
    // reference ctor tables (ORBextractor.cc:410-470)
    std::vector<float> scale, inv_scale, sigma2, inv_sigma2;
    std::vector<int> per_level;
    int umax[16];
    // geometry + workspace for the current (w,h)
    bool have_geom = false;
    borb::Geometry geom;
    borb::Workspace ws;
    int last_n_images = 0;       // images of the last batch (0: none)
    int in_channels = 1;         // host input pixel format (borb_extractor_set_input_format): 1 gray, 3 RGB/BGR, 4 RGBA/BGRA
    int in_rgb = 1;              // 1: R first (mbRGB), 0: B first
    // rectification maps (borb_extractor_set_rectify_maps): set 0 = mono / left, set 1 = right; device float maps
    float* d_map[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
    int map_src_w = 0, map_src_h = 0, map_dst_w = 0, map_dst_h = 0;
    int fast_mode = 0;           // fast_kernel ablation mode (borb_debug_set_fast_mode)
    uint64_t launches = 0;
    // stage timing: a ring of event sets so that many queued steps can be timed without host syncs
    static constexpr int EV_RING = 128;
    bool timing = false;
    std::vector<cudaEvent_t> ev;          // EV_RING * 9, created lazily
    unsigned ev_mask[EV_RING] = {};       // which of the 9 marks were recorded in that slot
    int ev_slot = 0;                      // slot of the step being enqueued
    int ev_pending = 0;                   // steps enqueued since the last borb_sync
    float stage_ms[8] = {};               // last step
    double stage_sum_ms[8] = {};          // accumulated since borb_set_timing(1)
    uint64_t stage_steps = 0;
    // staging
    int* h_counts = nullptr;     // pinned staging for the stereo pair table (2 ints per image)
    std::vector<int> pair_cache; // pair table currently resident in ws.pair_idx
};
