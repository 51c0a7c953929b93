// pcl_kernels.cuh — kernel parameter blocks + launch prototypes.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pcl.h"

namespace pcl {

struct CropParams {
  int B, H, W, pitch, S;
  pcl_crop_spec crop;
  const int32_t* sprites;
  int32_t* plot;
  int32_t* state;                // i32 [B, 4] per-cropper corner state, or NULL
  const uint8_t* board;
  uint8_t* out;
  const uint8_t* curtains[PCL_MAX_TRACK];   // byte curtains of tracked drapes (or NULL)
  uint32_t cols_recip;           // floor(2^32 / crop.cols) + 1, set by the launcher
};

// Everything a fused step kernel needs, by value (fits the 4 KB param space).
struct StepParams {
  int B, H, W, pitch;
  int PH, PW, PWW;               // Scrolly pattern rows/cols/words-per-row
  int BW;                        // words per bit-packed board-sized row
  int S, D;
  int auto_reset;
  int mode;                      // MODE_STEP / MODE_RESET
  int actions_per_env;
  int margin[PCL_MAX_DRAPES][2];
  uint8_t sprite_char[PCL_MAX_SPRITES];
  uint8_t drape_char[PCL_MAX_DRAPES];
  uint32_t impassable[PCL_MAX_SPRITES][4];
  int confined[PCL_MAX_SPRITES];
  int egocentric[PCL_MAX_SPRITES];
  int drape_kind[PCL_MAX_DRAPES];
  int program_arg[8];
  int n_scroll_groups;
  int sprite_group[PCL_MAX_SPRITES];
  int drape_group[PCL_MAX_DRAPES];
  int n_groups;
  int group_len[PCL_MAX_SPRITES + PCL_MAX_DRAPES];
  uint8_t group_chars[PCL_MAX_SPRITES + PCL_MAX_DRAPES];
  pcl_state st;
  pcl_outputs out;
  const int32_t* actions;        // i32 [B, actions_per_env] (MODE_STEP)
  const uint8_t* env_mask;       // u8 [B] or NULL (MODE_RESET)
  int has_cropper;               // pcl_attach_cropper: crop the new board as the kernel's epilogue
  CropParams cropper;            // (board is taken from `out` at launch time)
};

cudaError_t launch_scrolly_maze(const StepParams& p, cudaStream_t s);
cudaError_t launch_warehouse(const StepParams& p, cudaStream_t s);
cudaError_t launch_marauders(const StepParams& p, cudaStream_t s);
cudaError_t launch_fixture(const StepParams& p, cudaStream_t s);
cudaError_t launch_better_scrolly(const StepParams& p, cudaStream_t s);
cudaError_t launch_classics(const StepParams& p, cudaStream_t s);
cudaError_t launch_aperture(const StepParams& p, cudaStream_t s);
cudaError_t launch_ordeal(const StepParams& p, cudaStream_t s);
cudaError_t launch_hello(const StepParams& p, cudaStream_t s);
cudaError_t launch_apprehend(const StepParams& p, cudaStream_t s);
cudaError_t launch_shockwave(const StepParams& p, cudaStream_t s);
cudaError_t launch_box_world(const StepParams& p, cudaStream_t s);

struct RenderParams {
  int B, H, W, pitch, S, D;
  const uint8_t* backdrop; int64_t backdrop_bstride;
  const uint8_t* curtains;       // u8 [B, D, H, pitch]
  const int32_t* sprites;        // i32 [B, S, 8]
  const uint8_t* z_order;        // u8 [B, S + D] chars
  uint8_t sprite_char[PCL_MAX_SPRITES];
  uint8_t drape_char[PCL_MAX_DRAPES];
  uint8_t* board;                // u8 [B, H, pitch]
};
cudaError_t launch_render(const RenderParams& p, cudaStream_t s);

struct ExportParams {
  int B, H, W, pitch, PWW, BW, drape, scrolly;
  const uint32_t* bits; int64_t bits_bstride;   // pattern (scrolly) or board bits
  const int32_t* level;          // level index when `bits` is per-level static data, else NULL
  const int32_t* drapes; int D;
  int stale_slot;                // drape aux pair holding a stale cell, or -1
  uint8_t* out;
};
cudaError_t launch_export_curtain(const ExportParams& p, cudaStream_t s);

// Unoccluded layers (rendering.py:187-301): one mask per requested character.
#define PCL_MAX_LAYER_CHARS 32
struct LayersParams {
  int B, H, W, pitch, S, D, n_chars;
  uint8_t chars[PCL_MAX_LAYER_CHARS];
  int8_t sprite_of[PCL_MAX_LAYER_CHARS];   // sprite index painting that char, or -1
  int8_t drape_of[PCL_MAX_LAYER_CHARS];    // drape index painting that char, or -1
  // per drape: where its curtain lives in the packed state (as ExportParams)
  const uint32_t* bits[PCL_MAX_DRAPES]; int64_t bits_bstride[PCL_MAX_DRAPES];
  int row_words[PCL_MAX_DRAPES];           // uint32 words per bit row
  int scrolly[PCL_MAX_DRAPES];             // 1: window of a pattern at the drape's corner
  int per_level[PCL_MAX_DRAPES];           // 1: `bits` is static per-level data
  int stale_slot[PCL_MAX_DRAPES];          // 1: the drape record's AUX0/1 hold a stale cell
  const uint8_t* backdrop; int64_t backdrop_bstride;
  const int32_t* level;
  const int32_t* sprites;
  const int32_t* drapes;
  uint8_t* out;                            // u8 [B, n_chars, H, pitch]
};
cudaError_t launch_layers(const LayersParams& p, cudaStream_t s);

struct ObserveParams {
  int B, H, W, pitch, depth, dtype;
  int words;                     // 32-bit words per element (2 for int64 / float64)
  int64_t stride_b, stride_d, stride_r, stride_c;   // in 32-bit words (bytes for uint8)
  const void* table;             // [128, depth]
  const uint8_t* valid;          // u8 [128] or NULL
  const uint8_t* board;          // u8 [B, H, pitch]
  void* out;
  int32_t* unknown;              // i32 [1] or NULL
};
cudaError_t launch_observe(const ObserveParams& p, cudaStream_t s);

cudaError_t launch_crop(const CropParams& p, cudaStream_t s);

// Exchange state of the fused crop + hand-off kernel (pcl_crop_handoff).
struct HandoffParams {
  int n_peers, rank, record_bytes;
  int64_t rows;                  // records per half of a gather buffer
  int64_t first_row;             // this rank's first row
  uint8_t* peer_base[PCL_MAX_PEERS];    // peer-mapped bases of every rank's gather buffer (2 halves)
  uint32_t* peer_flags[PCL_MAX_PEERS];  // peer-mapped flag arrays u32 [PCL_MAX_PEERS] of every rank
  uint8_t* multicast;            // NVLS multicast mapping of the gather buffers, or NULL
  uint32_t* local;               // device-local u32 [2]: steps done, block ticket
  int n_bufs, lag;               // parts of the gather buffer; 1 = wait for the previous step only
  int signal_kernel;             // 1: a second one-warp kernel publishes and waits (no fences here)
  pcl_outputs out;
};
cudaError_t launch_crop_handoff(const CropParams& p, const HandoffParams& x, cudaStream_t s);

struct PackParams {
  int B, view_bytes, record_bytes;
  const uint8_t* view;           // u8 [B, view_bytes]
  pcl_outputs out;
  uint8_t* packed;               // u8 [B, record_bytes] (n_peers == 0)
  int n_peers;                   // > 0: store into every peer's gather buffer instead
  int64_t first_row;
  uint8_t* peers[PCL_MAX_PEERS];
};
cudaError_t launch_pack_handoff(const PackParams& p, cudaStream_t s);

}  // namespace pcl
