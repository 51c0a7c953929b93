// api.cu — the extern "C" boundary declared in include/pcl.h.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <new>

#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: ranges show up in nsys / ncu timelines

#include "pcl_device.cuh"
#include "pcl_kernels.cuh"


struct pcl_handle {
  pcl_spec spec;
  int batch;
  int device;
  int bound;
  int actions_per_env;
  pcl_state st;
  long long launches;
  pcl::StepParams base;          // everything fill_params derives from spec + state, built once at bind
  char last_error[256];          // text of the last failed CUDA call (pcl_last_error)
  // pcl_step_host_async: a copy stream so that the D2H of one step overlaps the next kernel
  cudaStream_t copy_stream;
  cudaEvent_t ev_step[PCL_HOST_SLOTS];   // step kernel finished (compute stream)
  cudaEvent_t ev_done[PCL_HOST_SLOTS];   // host buffers of that slot are valid (copy stream)
  int host_ready;
  int pending_slot;              // slot of this handle's last async step whose D2H may still run, or -1
};

namespace {

using pcl::StepParams;

// One NVTX range per boundary call (a no-op costing a pointer test when no tool
// is attached); the ranges name the reference call each entry point stands for.
struct Range {
  explicit Range(const char* name) { nvtxRangePushA(name); }
  ~Range() { nvtxRangePop(); }
};

// Remember what failed: PCL_ERR_CUDA alone says nothing (pcl_last_error).
int cuda_failed(pcl_handle* h, cudaError_t e, const char* what) {
  if (h) snprintf(h->last_error, sizeof(h->last_error), "%s: %s (%s)", what,
                  cudaGetErrorString(e), cudaGetErrorName(e));
  return PCL_ERR_CUDA;
}

#define PCL_CUDA(h, call)                                        \
  do {                                                           \
    cudaError_t e_ = (call);                                     \
    if (e_ != cudaSuccess) return cuda_failed((h), e_, #call);   \
  } while (0)

bool chars_are(const uint8_t* got, int n, const char* want) {
  if ((int)strlen(want) != n) return false;
  for (int i = 0; i < n; ++i) if (got[i] != (uint8_t)want[i]) return false;
  return true;
}

// The set `want` as a 128-bit ASCII mask equals `got`?
bool set_is(const uint32_t (&got)[4], const char* want) {
  uint32_t m[4] = {0, 0, 0, 0};
  for (const char* c = want; *c; ++c) m[(*c >> 5) & 3] |= 1u << (*c & 31);
  return m[0] == got[0] && m[1] == got[1] && m[2] == got[2] && m[3] == got[3];
}

int groups_are(const pcl_spec& s, const char* flat, const int* lens, int n) {
  if (s.n_groups != n) return 0;
  int k = 0;
  for (int g = 0; g < n; ++g) {
    if (s.group_len[g] != lens[g]) return 0;
    for (int i = 0; i < lens[g]; ++i, ++k)
      if (s.group_chars[k] != (uint8_t)flat[k]) return 0;
  }
  return 1;
}

// Each program is lowered for one entity layout; anything else is a valid
// pycolab game that this build does not accelerate.
int validate(const pcl_spec& s) {
  if (s.abi_version != PCL_ABI_VERSION) return PCL_ERR_INVALID;
  if (s.rows <= 0 || s.cols <= 0 || s.pitch < s.cols || (s.pitch & 15)) return PCL_ERR_INVALID;
  if (s.n_sprites < 0 || s.n_sprites > PCL_MAX_SPRITES) return PCL_ERR_INVALID;
  if (s.n_drapes < 0 || s.n_drapes > PCL_MAX_DRAPES) return PCL_ERR_INVALID;
  {
    // Scrolling groups: every entity names one of the declared groups; only the
    // general program keeps more than one group's blackboard.
    const int ng = s.n_scroll_groups < 1 ? 1 : s.n_scroll_groups;
    if (ng > PCL_MAX_SCROLL_GROUPS) return PCL_ERR_UNSUPPORTED;
    if (ng > 1 && s.program != PCL_PROG_FIXTURE) return PCL_ERR_UNSUPPORTED;
    for (int i = 0; i < s.n_sprites; ++i)
      if (s.sprite_group[i] < 0 || s.sprite_group[i] >= ng) return PCL_ERR_INVALID;
    for (int i = 0; i < s.n_drapes; ++i)
      if (s.drape_group[i] < 0 || s.drape_group[i] >= ng) return PCL_ERR_INVALID;
  }
  switch (s.program) {
    case PCL_PROG_NONE:
      return PCL_OK;
    case PCL_PROG_SCROLLY_MAZE: {
      if (!chars_are(s.sprite_char, s.n_sprites, "Pabc")) return PCL_ERR_UNSUPPORTED;
      if (!chars_are(s.drape_char, s.n_drapes, "#@")) return PCL_ERR_UNSUPPORTED;
      if (!chars_are(s.z_order, 6, "abc@#P")) return PCL_ERR_UNSUPPORTED;
      const int lens[3] = {1, 4, 1};
      if (!groups_are(s, "#abcP@", lens, 3)) return PCL_ERR_UNSUPPORTED;
      for (int i = 0; i < 4; ++i) {
        if (!set_is(s.impassable[i], "#")) return PCL_ERR_UNSUPPORTED;
        if (s.sprite_confined[i]) return PCL_ERR_UNSUPPORTED;
        if (s.sprite_egocentric[i] != (i == 0)) return PCL_ERR_UNSUPPORTED;
      }
      if (s.pattern_rows < s.rows || s.pattern_cols < s.cols) return PCL_ERR_INVALID;
      {
        // Window rows are staged from the even word at or below corner_c >> 5:
        // 2 * ceil((63 + W) / 64) words (4 up to 64 columns) must stay inside the row.
        const int nw = 2 * ((63 + s.cols + 63) / 64);
        if ((s.pattern_words & 1) || s.pattern_words < (((s.pattern_cols - s.cols) >> 5) & ~1) + nw ||
            s.pattern_words < (s.pattern_cols + 31) / 32 + 1) return PCL_ERR_INVALID;
        // one CTA (4 envs) stages tile + windows in shared memory
        const long per_env = 256L + (long)s.rows * s.pitch + 2L * s.rows * nw * 4 +
                             (long)s.rows * (s.pitch >> 2) + 64;
        if (per_env * 4 > 227L * 1024) return PCL_ERR_UNSUPPORTED;
      }
      for (int d = 0; d < 2; ++d) {
        const int mr = s.margins[d][0], mc = s.margins[d][1];
        if (mr >= 0 && (mc - 1 >= s.cols - mc || mr - 1 >= s.rows - mr)) return PCL_ERR_INVALID;
      }
      return PCL_OK;
    }
    case PCL_PROG_WAREHOUSE: {
      const int nb = s.n_sprites - 1;
      if (nb < 1 || nb > 10) return PCL_ERR_UNSUPPORTED;
      if (s.sprite_char[nb] != 'P') return PCL_ERR_UNSUPPORTED;
      if (!chars_are(s.drape_char, s.n_drapes, "X")) return PCL_ERR_UNSUPPORTED;
      const char* order = "1234567890";
      int k = 0;
      for (int i = 0; i < nb; ++i) {
        while (order[k] && order[k] != (char)s.sprite_char[i]) ++k;
        if (!order[k]) return PCL_ERR_UNSUPPORTED;
        ++k;
        if (s.z_order[i] != s.sprite_char[i]) return PCL_ERR_UNSUPPORTED;
        if (s.sprite_confined[i] || s.sprite_egocentric[i]) return PCL_ERR_UNSUPPORTED;
      }
      if (s.z_order[nb] != 'X' || s.z_order[nb + 1] != 'P') return PCL_ERR_UNSUPPORTED;
      if (s.n_groups != 3 || s.group_len[0] != nb || s.group_len[1] != 1 || s.group_len[2] != 1)
        return PCL_ERR_UNSUPPORTED;
      for (int i = 0; i < nb; ++i)
        if (s.group_chars[i] != s.sprite_char[i]) return PCL_ERR_UNSUPPORTED;
      if (s.group_chars[nb] != 'X' || s.group_chars[nb + 1] != 'P') return PCL_ERR_UNSUPPORTED;
      return PCL_OK;
    }
    case PCL_PROG_MARAUDERS: {
      if (!chars_are(s.sprite_char, s.n_sprites, "Pabcdyz")) return PCL_ERR_UNSUPPORTED;
      if (!chars_are(s.drape_char, s.n_drapes, "BX")) return PCL_ERR_UNSUPPORTED;
      if (!chars_are(s.z_order, 9, "PBXabcdyz")) return PCL_ERR_UNSUPPORTED;
      const int lens[1] = {9};
      if (!groups_are(s, "PBXabcdyz", lens, 1)) return PCL_ERR_UNSUPPORTED;
      if (s.rows > 32 || s.rows < 11 || s.cols > 64 || s.bits_words < 2)
        return PCL_ERR_UNSUPPORTED;
      for (int i = 0; i < 7; ++i) {
        if (!set_is(s.impassable[i], "")) return PCL_ERR_UNSUPPORTED;
        if (s.sprite_confined[i] != (i == 0) || s.sprite_egocentric[i]) return PCL_ERR_UNSUPPORTED;
      }
      return PCL_OK;
    }
    case PCL_PROG_BETTER_SCROLLY: {
      if (!chars_are(s.sprite_char, s.n_sprites, "Pabc")) return PCL_ERR_UNSUPPORTED;
      if (!chars_are(s.drape_char, s.n_drapes, "@")) return PCL_ERR_UNSUPPORTED;
      if (!chars_are(s.z_order, 5, "abc@P")) return PCL_ERR_UNSUPPORTED;
      const int lens[1] = {5};
      if (!groups_are(s, "abcP@", lens, 1)) return PCL_ERR_UNSUPPORTED;
      for (int i = 0; i < 4; ++i)
        if (s.sprite_confined[i] || s.sprite_egocentric[i]) return PCL_ERR_UNSUPPORTED;
      if (s.bits_words < (s.cols + 31) / 32 + 1) return PCL_ERR_INVALID;
      return PCL_OK;
    }
    case PCL_PROG_CLASSICS: {
      if (!chars_are(s.sprite_char, s.n_sprites, "P") || s.n_drapes != 0) return PCL_ERR_UNSUPPORTED;
      if (!chars_are(s.z_order, 1, "P")) return PCL_ERR_UNSUPPORTED;
      const int lens[1] = {1};
      if (!groups_are(s, "P", lens, 1)) return PCL_ERR_UNSUPPORTED;
      if (s.sprite_egocentric[0]) return PCL_ERR_UNSUPPORTED;
      const int rule = s.program_arg[0];
      if (rule != PCL_CLASSIC_FOUR_ROOMS && rule != PCL_CLASSIC_CLIFF_WALK &&
          rule != PCL_CLASSIC_CHAIN_WALK && rule != PCL_CLASSIC_FLUVIAL) return PCL_ERR_INVALID;
      if (rule == PCL_CLASSIC_FLUVIAL) {
        // The kernel re-stages the flowing rows before the swimmer moves, which is
        // only equivalent when the swimmer never looks at the board.
        if (!set_is(s.impassable[0], "")) return PCL_ERR_UNSUPPORTED;
        if (s.program_arg[1] < 0 || s.program_arg[2] < s.program_arg[1]) return PCL_ERR_INVALID;
      }
      if (s.rows * s.pitch > 8192) return PCL_ERR_UNSUPPORTED;   // the tile is staged per env in smem
      return PCL_OK;
    }
    case PCL_PROG_APERTURE: {
      if (s.n_sprites != 1 || s.n_drapes != 1) return PCL_ERR_UNSUPPORTED;
      if (s.z_order[0] != s.drape_char[0] || s.z_order[1] != s.sprite_char[0]) return PCL_ERR_UNSUPPORTED;
      if (s.n_groups != 2 || s.group_len[0] != 1 || s.group_len[1] != 1 ||
          s.group_chars[0] != s.sprite_char[0] || s.group_chars[1] != s.drape_char[0])
        return PCL_ERR_UNSUPPORTED;
      if (s.sprite_egocentric[0]) return PCL_ERR_UNSUPPORTED;
      if (s.rows >= 32768 || s.cols >= 32768 || s.rows * s.pitch > 8192) return PCL_ERR_UNSUPPORTED;
      return PCL_OK;
    }
    case PCL_PROG_HELLO: {
      if (s.n_sprites < 1 || s.n_sprites > 4 || s.n_drapes != 1) return PCL_ERR_UNSUPPORTED;
      if (s.n_groups != 1 || s.group_len[0] != s.n_sprites + 1) return PCL_ERR_UNSUPPORTED;
      if (s.bits_words < (s.cols + 31) / 32 + 1) return PCL_ERR_INVALID;
      for (int k = 0; k < s.n_sprites + 1; ++k)      // program_arg = the z-order
        if (s.program_arg[k] != s.z_order[k]) return PCL_ERR_INVALID;
      return PCL_OK;
    }
    case PCL_PROG_APPREHEND: {
      if (s.n_sprites != 2 || s.n_drapes != 0) return PCL_ERR_UNSUPPORTED;
      // one update group: the ball, then the catcher; the catcher is drawn on top
      if (s.n_groups != 1 || s.group_len[0] != 2 || s.group_chars[0] != s.sprite_char[1] ||
          s.group_chars[1] != s.sprite_char[0]) return PCL_ERR_UNSUPPORTED;
      if (s.z_order[0] != s.sprite_char[1] || s.z_order[1] != s.sprite_char[0]) return PCL_ERR_UNSUPPORTED;
      if (!s.sprite_confined[0] || s.sprite_confined[1]) return PCL_ERR_UNSUPPORTED;
      for (int i = 0; i < 2; ++i) {
        if (s.sprite_egocentric[i]) return PCL_ERR_UNSUPPORTED;
        for (int w = 0; w < 4; ++w) if (s.impassable[i][w]) return PCL_ERR_UNSUPPORTED;
      }
      if (s.rows < 2) return PCL_ERR_INVALID;          // the slope divides by rows - 1
      return PCL_OK;
    }
    case PCL_PROG_SHOCKWAVE: {
      if (s.n_sprites != 1 || s.n_drapes != 3) return PCL_ERR_UNSUPPORTED;
      // one update group [' ', '^', P, '@'] (the two static drapes may come in either
      // order), z-order ' ' '^' '@' P
      if (s.n_groups != 1 || s.group_len[0] != 4 || s.group_chars[2] != s.sprite_char[0] ||
          s.group_chars[3] != s.drape_char[0]) return PCL_ERR_UNSUPPORTED;
      if (s.z_order[0] != s.drape_char[1] || s.z_order[1] != s.drape_char[2] ||
          s.z_order[2] != s.drape_char[0] || s.z_order[3] != s.sprite_char[0]) return PCL_ERR_UNSUPPORTED;
      if (!s.sprite_confined[0] || s.sprite_egocentric[0]) return PCL_ERR_UNSUPPORTED;
      if (s.rows > 32 || s.cols > 64) return PCL_ERR_UNSUPPORTED;      // a curtain row per lane, 64-bit rows
      if (s.bits_words < (s.cols + 31) / 32 + 1) return PCL_ERR_INVALID;
      if (s.program_arg[0] < 0 || s.program_arg[0] > 1024) return PCL_ERR_INVALID;
      return PCL_OK;
    }
    case PCL_PROG_ORDEAL: {
      const int chapter = s.program_arg[0];
      const int want_s = chapter == PCL_ORDEAL_CASTLE ? 2 : 1, want_d = chapter == PCL_ORDEAL_CAVERN ? 1 : 0;
      if (chapter != PCL_ORDEAL_CASTLE && chapter != PCL_ORDEAL_CAVERN && chapter != PCL_ORDEAL_KANSAS)
        return PCL_ERR_INVALID;
      if (s.n_sprites != want_s || s.n_drapes != want_d) return PCL_ERR_UNSUPPORTED;
      if (s.n_groups != 1 || s.group_len[0] != want_s + want_d) return PCL_ERR_UNSUPPORTED;
      if (s.group_chars[0] != s.sprite_char[0]) return PCL_ERR_UNSUPPORTED;     // the player moves first
      for (int i = 0; i < want_s; ++i) if (s.sprite_egocentric[i]) return PCL_ERR_UNSUPPORTED;
      if (s.rows >= 32768 || s.cols >= 32768 || s.rows * s.pitch > 8192) return PCL_ERR_UNSUPPORTED;
      if (want_d && s.bits_words < (s.cols + 31) / 32 + 1) return PCL_ERR_INVALID;
      return PCL_OK;
    }
    case PCL_PROG_BOX_WORLD: {
      // The player alone is an entity of the spec; the drapes live in the cell plane.
      if (s.n_sprites != 1 || s.n_drapes != 0) return PCL_ERR_UNSUPPORTED;
      const int lens[1] = {1};
      if (!groups_are(s, (const char*)s.sprite_char, lens, 1) || s.z_order[0] != s.sprite_char[0])
        return PCL_ERR_UNSUPPORTED;
      if (!s.sprite_confined[0] || s.sprite_egocentric[0] || !set_is(s.impassable[0], "#"))
        return PCL_ERR_UNSUPPORTED;
      // a plane of at most 64 16-byte row segments: two per lane of the env's warp
      if (s.rows > 32 || s.cols > 32 || s.pitch > 32) return PCL_ERR_UNSUPPORTED;
      if (s.rows < 3 || s.cols < 3 || s.bits_words * 4 != s.pitch) return PCL_ERR_INVALID;
      const int stride = s.program_arg[1], levels = s.program_arg[2];
      if (stride < 0 || levels < 0 || (stride > 0 && levels < 1)) return PCL_ERR_INVALID;
      return PCL_OK;
    }
    case PCL_PROG_FIXTURE: {
      // Any MazeWalker / Scrolly / plain-drape mix; entities and z-order must
      // be consistent permutations of each other.
      const int n = s.n_sprites + s.n_drapes;
      if (n < 1) return PCL_ERR_INVALID;
      int total = 0;
      for (int g = 0; g < s.n_groups; ++g) total += s.group_len[g];
      if (s.n_groups < 1 || total != n) return PCL_ERR_INVALID;
      for (int i = 0; i < n; ++i) {
        int in_z = 0, in_groups = 0;
        const uint8_t ch = i < s.n_sprites ? s.sprite_char[i] : s.drape_char[i - s.n_sprites];
        for (int k = 0; k < n; ++k) {
          in_z += s.z_order[k] == ch;
          in_groups += s.group_chars[k] == ch;
        }
        if (in_z != 1 || in_groups != 1 || ch == 0 || ch > 127) return PCL_ERR_INVALID;
      }
      for (int d = 0; d < s.n_drapes; ++d) {
        if (!s.drape_kind[d]) continue;
        if (s.pattern_rows < s.rows || s.pattern_cols < s.cols) return PCL_ERR_INVALID;
        if (s.pattern_words < (s.pattern_cols + 31) / 32 + 2) return PCL_ERR_INVALID;
        const int mr = s.margins[d][0], mc = s.margins[d][1];
        if (mr >= 0 && (mc - 1 >= s.cols - mc || mr - 1 >= s.rows - mr)) return PCL_ERR_INVALID;
      }
      if (s.bits_words < (s.cols + 31) / 32 + 1) return PCL_ERR_INVALID;
      return PCL_OK;
    }
    default:
      return PCL_ERR_UNSUPPORTED;
  }
}

void fill_params(const pcl_handle* h, StepParams* p) {
  const pcl_spec& s = h->spec;
  memset(p, 0, sizeof(*p));
  p->B = h->batch; p->H = s.rows; p->W = s.cols; p->pitch = s.pitch;
  p->PH = s.pattern_rows; p->PW = s.pattern_cols; p->PWW = s.pattern_words;
  p->BW = s.bits_words;
  p->S = s.n_sprites; p->D = s.n_drapes;
  p->auto_reset = s.auto_reset;
  p->actions_per_env = h->actions_per_env;
  memcpy(p->margin, s.margins, sizeof(p->margin));
  memcpy(p->sprite_char, s.sprite_char, sizeof(p->sprite_char));
  memcpy(p->drape_char, s.drape_char, sizeof(p->drape_char));
  memcpy(p->impassable, s.impassable, sizeof(p->impassable));
  memcpy(p->confined, s.sprite_confined, sizeof(p->confined));
  memcpy(p->egocentric, s.sprite_egocentric, sizeof(p->egocentric));
  memcpy(p->drape_kind, s.drape_kind, sizeof(p->drape_kind));
  memcpy(p->program_arg, s.program_arg, sizeof(p->program_arg));
  p->n_scroll_groups = s.n_scroll_groups < 1 ? 1 : s.n_scroll_groups;
  memcpy(p->sprite_group, s.sprite_group, sizeof(p->sprite_group));
  memcpy(p->drape_group, s.drape_group, sizeof(p->drape_group));
  p->n_groups = s.n_groups;
  memcpy(p->group_len, s.group_len, sizeof(p->group_len));
  memcpy(p->group_chars, s.group_chars, sizeof(p->group_chars));
  p->st = h->st;
}

int launch(pcl_handle* h, const StepParams& p, cudaStream_t stream) {
  cudaError_t e;
  switch (h->spec.program) {
    case PCL_PROG_SCROLLY_MAZE: e = pcl::launch_scrolly_maze(p, stream); break;
    case PCL_PROG_WAREHOUSE: e = pcl::launch_warehouse(p, stream); break;
    case PCL_PROG_MARAUDERS: e = pcl::launch_marauders(p, stream); break;
    case PCL_PROG_FIXTURE: e = pcl::launch_fixture(p, stream); break;
    case PCL_PROG_BETTER_SCROLLY: e = pcl::launch_better_scrolly(p, stream); break;
    case PCL_PROG_CLASSICS: e = pcl::launch_classics(p, stream); break;
    case PCL_PROG_APERTURE: e = pcl::launch_aperture(p, stream); break;
    case PCL_PROG_ORDEAL: e = pcl::launch_ordeal(p, stream); break;
    case PCL_PROG_HELLO: e = pcl::launch_hello(p, stream); break;
    case PCL_PROG_APPREHEND: e = pcl::launch_apprehend(p, stream); break;
    case PCL_PROG_SHOCKWAVE: e = pcl::launch_shockwave(p, stream); break;
    case PCL_PROG_BOX_WORLD: e = pcl::launch_box_world(p, stream); break;
    default: return PCL_ERR_UNSUPPORTED;
  }
  if (e != cudaSuccess) return cuda_failed(h, e, "step kernel launch");
  h->launches += 1;              // only launches that were accepted count
  return PCL_OK;
}

// Status of a non-step kernel launch; counts it when it went through.
int launched(pcl_handle* h, cudaError_t e, const char* what) {
  if (e != cudaSuccess) return cuda_failed(h, e, what);
  h->launches += 1;
  return PCL_OK;
}

int check_ready(const pcl_handle* h, const pcl_outputs* out) {
  if (!h || !out) return PCL_ERR_INVALID;
  if (!h->bound) return PCL_ERR_UNBOUND;
  if (!out->d_board || !out->d_reward || !out->d_has_reward || !out->d_discount || !out->d_done)
    return PCL_ERR_INVALID;
  return PCL_OK;
}

__global__ void gather_errors(const int32_t* plot, int32_t* out, int B) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) out[i] = plot[(int64_t)i * PCL_PLOT_WORDS + PCL_P_ERROR];
}

}  // namespace

extern "C" {

int pcl_abi_version(void) { return PCL_ABI_VERSION; }

int pcl_struct_sizes(int32_t out[4]) {
  if (!out) return PCL_ERR_INVALID;
  out[0] = (int32_t)sizeof(pcl_spec); out[1] = (int32_t)sizeof(pcl_state);
  out[2] = (int32_t)sizeof(pcl_outputs); out[3] = (int32_t)sizeof(pcl_crop_spec);
  return PCL_OK;
}

const char* pcl_status_string(int status) {
  switch (status) {
    case PCL_OK: return "ok";
    case PCL_ERR_INVALID: return "invalid argument or malformed spec";
    case PCL_ERR_UNSUPPORTED: return "game not lowered to a device program";
    case PCL_ERR_CUDA: return "CUDA runtime error";
    case PCL_ERR_UNBOUND: return "pcl_bind_state has not been called";
    case PCL_ERR_NOMEM: return "out of memory";
    default: return "unknown status";
  }
}

int pcl_create(const pcl_spec* spec, int batch, int device, pcl_handle** out) {
  if (!spec || !out || batch <= 0) return PCL_ERR_INVALID;
  const int v = validate(*spec);
  if (v != PCL_OK) return v;
  if (device >= 0 && cudaSetDevice(device) != cudaSuccess) return PCL_ERR_CUDA;
  pcl_handle* h = new (std::nothrow) pcl_handle();
  if (!h) return PCL_ERR_NOMEM;
  h->spec = *spec;
  h->batch = batch;
  h->device = device;
  h->bound = 0;
  h->actions_per_env = spec->program == PCL_PROG_FIXTURE ? spec->n_sprites + spec->n_drapes + 2 * PCL_FIXTURE_DIRECTIVES : 1;
  h->launches = 0;
  h->last_error[0] = 0;
  h->host_ready = 0;
  h->pending_slot = -1;
  *out = h;
  return PCL_OK;
}

int pcl_destroy(pcl_handle* h) {
  if (h && h->host_ready) {
    for (int i = 0; i < PCL_HOST_SLOTS; ++i) {
      cudaEventDestroy(h->ev_step[i]);
      cudaEventDestroy(h->ev_done[i]);
    }
    cudaStreamDestroy(h->copy_stream);
  }
  delete h;
  return PCL_OK;
}

const char* pcl_last_error(pcl_handle* h) { return h ? h->last_error : ""; }

int pcl_bind_state(pcl_handle* h, const pcl_state* st) {
  if (!h || !st) return PCL_ERR_INVALID;
  if (!st->d_backdrop || !st->d_plot || !st->d_plot_init) return PCL_ERR_INVALID;
  // A game may have no sprites at all (engine_test.py:578-640 renders one drape).
  if (h->spec.n_sprites > 0 && (!st->d_sprites || !st->d_sprites_init)) return PCL_ERR_INVALID;
  if (h->spec.n_drapes > 0 && (!st->d_drapes || !st->d_drapes_init)) return PCL_ERR_INVALID;
  if (h->spec.program == PCL_PROG_SCROLLY_MAZE) {
    for (int d = 0; d < 2; ++d) if (!st->d_pattern[d]) return PCL_ERR_INVALID;
    if (!st->d_pattern_init[1] || st->pattern_bstride[1] == 0) return PCL_ERR_INVALID;
  }
  if (h->spec.program == PCL_PROG_MARAUDERS) {
    for (int d = 0; d < 2; ++d)
      if (!st->d_bits[d] || !st->d_bits_init[d] || st->bits_bstride[d] == 0) return PCL_ERR_INVALID;
    if (!st->d_rng) return PCL_ERR_INVALID;
  }
  if (h->spec.program == PCL_PROG_HELLO && !st->d_bits_init[0]) return PCL_ERR_INVALID;
  if (h->spec.program == PCL_PROG_SHOCKWAVE) {
    if (!st->d_bits[0] || st->bits_bstride[0] == 0 || !st->d_rng) return PCL_ERR_INVALID;
    for (int d = 0; d < 3; ++d) if (!st->d_bits_init[d]) return PCL_ERR_INVALID;
  }
  if (h->spec.program == PCL_PROG_ORDEAL) {
    if (h->spec.n_drapes && (!st->d_bits[0] || !st->d_bits_init[0] || st->bits_bstride[0] == 0))
      return PCL_ERR_INVALID;
    if (h->spec.n_sprites + h->spec.n_drapes == 2 && (!st->d_z_order || !st->d_z_order_init))
      return PCL_ERR_INVALID;                   // the kernel reads the z-order of two entities
  }
  if (h->spec.program == PCL_PROG_BETTER_SCROLLY) {
    if (!st->d_bits[0] || !st->d_bits_init[0] || st->bits_bstride[0] == 0) return PCL_ERR_INVALID;
  }
  if (h->spec.program == PCL_PROG_BOX_WORLD) {
    if (!st->d_bits[0] || !st->d_bits_init[0] || st->bits_bstride[0] == 0) return PCL_ERR_INVALID;
    if (h->spec.program_arg[1] > 0 && !st->d_level) return PCL_ERR_INVALID;   // rotation writes it
  }
  if (h->spec.n_scroll_groups > 1 && (!st->d_groups || !st->d_groups_init)) return PCL_ERR_INVALID;
  if (h->spec.program == PCL_PROG_FIXTURE) {
    if (!st->d_z_order || !st->d_z_order_init) return PCL_ERR_INVALID;
    for (int d = 0; d < h->spec.n_drapes; ++d) {
      if (h->spec.drape_kind[d] ? !st->d_pattern[d] : !st->d_bits[d]) return PCL_ERR_INVALID;
    }
  }
  h->st = *st;
  fill_params(h, &h->base);      // the per-step calls only patch mode / actions / outputs
  h->bound = 1;
  return PCL_OK;
}

int pcl_reset(pcl_handle* h, const uint8_t* d_env_mask, const pcl_outputs* out, void* stream) {
  Range nvtx_range("pcl_reset (Engine.its_showtime)");
  const int r = check_ready(h, out);
  if (r != PCL_OK) return r;
  StepParams p = h->base;
  p.mode = pcl::MODE_RESET;
  p.env_mask = d_env_mask;
  p.out = *out;
  return launch(h, p, (cudaStream_t)stream);
}

int pcl_step(pcl_handle* h, const int32_t* d_actions, const pcl_outputs* out, void* stream) {
  Range nvtx_range("pcl_step (Engine.play)");
  const int r = check_ready(h, out);
  if (r != PCL_OK) return r;
  if (!d_actions) return PCL_ERR_INVALID;
  StepParams p = h->base;
  p.mode = pcl::MODE_STEP;
  p.actions = d_actions;
  p.out = *out;
  return launch(h, p, (cudaStream_t)stream);
}

int pcl_run(pcl_handle* h, const int32_t* d_actions, int steps, const pcl_outputs* out,
            void* stream) {
  Range nvtx_range("pcl_run");
  const int r = check_ready(h, out);
  if (r != PCL_OK) return r;
  if (!d_actions || steps < 0) return PCL_ERR_INVALID;
  StepParams p = h->base;
  p.mode = pcl::MODE_STEP;
  p.out = *out;
  for (int t = 0; t < steps; ++t) {
    p.actions = d_actions + (int64_t)t * h->batch * h->actions_per_env;
    const int e = launch(h, p, (cudaStream_t)stream);
    if (e != PCL_OK) return e;
  }
  return PCL_OK;
}

int pcl_run_many(pcl_handle* const* handles, int n_handles, const int32_t* const* d_actions,
                 const pcl_outputs* const* outs, int steps, void* stream) {
  Range nvtx_range("pcl_run_many");
  if (!handles || !d_actions || !outs || n_handles < 1 || steps < 0) return PCL_ERR_INVALID;
  for (int i = 0; i < n_handles; ++i) {
    const int r = check_ready(handles[i], outs[i]);
    if (r != PCL_OK) return r;
  }
  for (int t = 0; t < steps; ++t) {
    if (!d_actions[t]) return PCL_ERR_INVALID;
    pcl_handle* h = handles[t % n_handles];
    StepParams p = h->base;
    p.mode = pcl::MODE_STEP;
    p.out = *outs[t % n_handles];
    p.actions = d_actions[t];
    const int e = launch(h, p, (cudaStream_t)stream);
    if (e != PCL_OK) return e;
  }
  return PCL_OK;
}

namespace {

// H2D of the action words, then the step, both on `s`.
int step_host_enqueue(pcl_handle* h, const int32_t* h_actions, int32_t* d_actions,
                      const pcl_outputs* out, cudaStream_t s) {
  const size_t B = (size_t)h->batch;
  PCL_CUDA(h, cudaMemcpyAsync(d_actions, h_actions, B * h->actions_per_env * sizeof(int32_t),
                              cudaMemcpyHostToDevice, s));
  return pcl_step(h, d_actions, out, (void*)s);
}

int copy_outputs(pcl_handle* h, const pcl_outputs* out, const uint8_t* d_view, size_t view_bytes,
                 uint8_t* h_view, int32_t* h_reward, uint8_t* h_has_reward, float* h_discount,
                 uint8_t* h_done, cudaStream_t s) {
  const size_t B = (size_t)h->batch;
  if (h_view) PCL_CUDA(h, cudaMemcpyAsync(h_view, d_view, view_bytes, cudaMemcpyDeviceToHost, s));
  if (h_reward) PCL_CUDA(h, cudaMemcpyAsync(h_reward, out->d_reward, B * 4, cudaMemcpyDeviceToHost, s));
  if (h_has_reward)
    PCL_CUDA(h, cudaMemcpyAsync(h_has_reward, out->d_has_reward, B, cudaMemcpyDeviceToHost, s));
  if (h_discount)
    PCL_CUDA(h, cudaMemcpyAsync(h_discount, out->d_discount, B * 4, cudaMemcpyDeviceToHost, s));
  if (h_done) PCL_CUDA(h, cudaMemcpyAsync(h_done, out->d_done, B, cudaMemcpyDeviceToHost, s));
  return PCL_OK;
}

int host_pipeline_ready(pcl_handle* h) {
  if (h->host_ready) return PCL_OK;
  PCL_CUDA(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < PCL_HOST_SLOTS; ++i) {
    PCL_CUDA(h, cudaEventCreateWithFlags(&h->ev_step[i], cudaEventDisableTiming));
    PCL_CUDA(h, cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming));
  }
  h->host_ready = 1;
  return PCL_OK;
}

}  // namespace

int pcl_step_host(pcl_handle* h, const int32_t* h_actions, int32_t* d_actions,
                  const pcl_outputs* out, uint8_t* h_board, int32_t* h_reward,
                  uint8_t* h_has_reward, float* h_discount, uint8_t* h_done, void* stream) {
  Range nvtx_range("pcl_step_host");
  const int r = check_ready(h, out);
  if (r != PCL_OK) return r;
  if (!h_actions || !d_actions) return PCL_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t plane = (size_t)h->spec.rows * h->spec.pitch;
  int e = step_host_enqueue(h, h_actions, d_actions, out, s);
  if (e != PCL_OK) return e;
  e = copy_outputs(h, out, out->d_board, (size_t)h->batch * plane, h_board, h_reward, h_has_reward,
                   h_discount, h_done, s);
  if (e != PCL_OK) return e;
  PCL_CUDA(h, cudaStreamSynchronize(s));
  return PCL_OK;
}

int pcl_step_host_async(pcl_handle* h, const int32_t* h_actions, int32_t* d_actions,
                        const pcl_outputs* out, const pcl_crop_spec* crop, uint8_t* d_crop,
                        int32_t* d_crop_state, uint8_t* h_view, int32_t* h_reward,
                        uint8_t* h_has_reward, float* h_discount, uint8_t* h_done, int slot,
                        void* stream) {
  Range nvtx_range("pcl_step_host_async");
  const int r = check_ready(h, out);
  if (r != PCL_OK) return r;
  if (!h_actions || !d_actions || slot < 0 || slot >= PCL_HOST_SLOTS) return PCL_ERR_INVALID;
  if (crop && !d_crop) return PCL_ERR_INVALID;
  int e = host_pipeline_ready(h);
  if (e != PCL_OK) return e;
  cudaStream_t s = (cudaStream_t)stream;
  // This step overwrites the device outputs: the D2H of this handle's previous
  // async step must have read them.  Other handles sharing `s` are not held up.
  if (h->pending_slot >= 0) PCL_CUDA(h, cudaStreamWaitEvent(s, h->ev_done[h->pending_slot], 0));
  e = step_host_enqueue(h, h_actions, d_actions, out, s);
  if (e != PCL_OK) return e;
  const uint8_t* d_view = out->d_board;
  size_t view_bytes = (size_t)h->batch * h->spec.rows * h->spec.pitch;
  if (crop) {                    // only the cropped view crosses PCIe
    // The same cropper attached to the handle (pcl_attach_cropper) has already run as
    // the step kernel's epilogue: nothing more to launch.
    const bool fused = h->base.has_cropper && h->base.cropper.out == d_crop &&
                       h->base.cropper.state == d_crop_state &&
                       memcmp(&h->base.cropper.crop, crop, sizeof(*crop)) == 0;
    e = fused ? PCL_OK : pcl_crop(h, crop, out->d_board, d_crop, d_crop_state, stream);
    if (e != PCL_OK) return e;
    d_view = d_crop;
    view_bytes = (size_t)h->batch * crop->rows * crop->cols;
  }
  PCL_CUDA(h, cudaEventRecord(h->ev_step[slot], s));
  PCL_CUDA(h, cudaStreamWaitEvent(h->copy_stream, h->ev_step[slot], 0));
  e = copy_outputs(h, out, d_view, view_bytes, h_view, h_reward, h_has_reward, h_discount, h_done,
                   h->copy_stream);
  if (e != PCL_OK) return e;
  PCL_CUDA(h, cudaEventRecord(h->ev_done[slot], h->copy_stream));
  h->pending_slot = slot;
  return PCL_OK;
}

int pcl_host_wait(pcl_handle* h, int slot) {
  if (!h || slot < 0 || slot >= PCL_HOST_SLOTS || !h->host_ready) return PCL_ERR_INVALID;
  PCL_CUDA(h, cudaEventSynchronize(h->ev_done[slot]));
  return PCL_OK;
}

int pcl_render(pcl_handle* h, const uint8_t* d_backdrop, int64_t backdrop_bstride,
               const uint8_t* d_curtains, const int32_t* d_sprites, const uint8_t* d_z_order,
               uint8_t* d_board, void* stream) {
  Range nvtx_range("pcl_render (Engine._render)");
  if (!h || !d_backdrop || !d_z_order || !d_board) return PCL_ERR_INVALID;
  if (h->spec.n_drapes > 0 && !d_curtains) return PCL_ERR_INVALID;
  if (h->spec.n_sprites > 0 && !d_sprites) return PCL_ERR_INVALID;
  pcl::RenderParams p;
  memset(&p, 0, sizeof(p));
  p.B = h->batch; p.H = h->spec.rows; p.W = h->spec.cols; p.pitch = h->spec.pitch;
  p.S = h->spec.n_sprites; p.D = h->spec.n_drapes;
  p.backdrop = d_backdrop; p.backdrop_bstride = backdrop_bstride;
  p.curtains = d_curtains; p.sprites = d_sprites; p.z_order = d_z_order; p.board = d_board;
  memcpy(p.sprite_char, h->spec.sprite_char, sizeof(p.sprite_char));
  memcpy(p.drape_char, h->spec.drape_char, sizeof(p.drape_char));
  return launched(h, pcl::launch_render(p, (cudaStream_t)stream), "launch_render");
}

int pcl_export_curtain(pcl_handle* h, int drape_index, uint8_t* d_out, void* stream) {
  if (!h || !d_out || drape_index < 0 || drape_index >= h->spec.n_drapes) return PCL_ERR_INVALID;
  if (!h->bound) return PCL_ERR_UNBOUND;
  pcl::ExportParams p;
  memset(&p, 0, sizeof(p));
  p.B = h->batch; p.H = h->spec.rows; p.W = h->spec.cols; p.pitch = h->spec.pitch;
  p.PWW = h->spec.pattern_words; p.BW = h->spec.bits_words;
  p.drape = drape_index; p.D = h->spec.n_drapes; p.drapes = h->st.d_drapes;
  p.out = d_out; p.stale_slot = -1;
  if (h->spec.program == PCL_PROG_SCROLLY_MAZE) {
    p.scrolly = 1;
    p.bits = h->st.d_pattern[drape_index];
    p.bits_bstride = h->st.pattern_bstride[drape_index];
    if (drape_index == 1) p.stale_slot = 0;
    else p.level = h->st.d_level;            // the wall pattern is read-only: per level
  } else if (h->spec.program == PCL_PROG_MARAUDERS ||
             h->spec.program == PCL_PROG_BETTER_SCROLLY || h->spec.program == PCL_PROG_ORDEAL ||
             h->spec.program == PCL_PROG_SHOCKWAVE ||
             (h->spec.program == PCL_PROG_FIXTURE && !h->spec.drape_kind[drape_index])) {
    p.scrolly = 0;
    p.bits = h->st.d_bits[drape_index];
    p.bits_bstride = h->st.bits_bstride[drape_index];
  } else if (h->spec.program == PCL_PROG_FIXTURE) {
    p.scrolly = 1;
    p.bits = h->st.d_pattern[drape_index];
    p.bits_bstride = h->st.pattern_bstride[drape_index];
    p.level = h->st.d_level;                 // fixture patterns are read-only: per level
  } else {
    return PCL_ERR_UNSUPPORTED;
  }
  return launched(h, pcl::launch_export_curtain(p, (cudaStream_t)stream), "launch_export_curtain");
}

int pcl_layers(pcl_handle* h, const uint8_t* chars, int32_t n_chars, uint8_t* d_out,
               void* stream) {
  Range nvtx_range("pcl_layers");
  if (!h || !chars || !d_out || n_chars < 1 || n_chars > PCL_MAX_LAYER_CHARS)
    return PCL_ERR_INVALID;
  if (!h->bound) return PCL_ERR_UNBOUND;
  const pcl_spec& sp = h->spec;
  if (sp.program == PCL_PROG_BOX_WORLD) return PCL_ERR_UNSUPPORTED;   // drapes held in the cell plane
  pcl::LayersParams p;
  memset(&p, 0, sizeof(p));
  p.B = h->batch; p.H = sp.rows; p.W = sp.cols; p.pitch = sp.pitch;
  p.S = sp.n_sprites; p.D = sp.n_drapes; p.n_chars = n_chars;
  p.backdrop = h->st.d_backdrop; p.backdrop_bstride = h->st.backdrop_bstride;
  p.level = h->st.d_level; p.sprites = h->st.d_sprites; p.drapes = h->st.d_drapes;
  p.out = d_out;
  for (int d = 0; d < sp.n_drapes; ++d) {
    // Where each program keeps a drape's curtain (as pcl_export_curtain).
    if (sp.program == PCL_PROG_SCROLLY_MAZE ||
        (sp.program == PCL_PROG_FIXTURE && sp.drape_kind[d])) {
      p.scrolly[d] = 1;
      p.bits[d] = h->st.d_pattern[d]; p.bits_bstride[d] = h->st.pattern_bstride[d];
      p.row_words[d] = sp.pattern_words;
      const bool coins = sp.program == PCL_PROG_SCROLLY_MAZE && d == 1;
      p.stale_slot[d] = coins;
      p.per_level[d] = !coins && h->st.d_level != nullptr;   // read-only patterns: per level
    } else if (sp.program == PCL_PROG_MARAUDERS || sp.program == PCL_PROG_BETTER_SCROLLY ||
               sp.program == PCL_PROG_FIXTURE || sp.program == PCL_PROG_ORDEAL ||
               sp.program == PCL_PROG_SHOCKWAVE) {
      p.bits[d] = h->st.d_bits[d]; p.bits_bstride[d] = h->st.bits_bstride[d];
      p.row_words[d] = sp.bits_words;
    } else {
      return PCL_ERR_UNSUPPORTED;       // curtain held implicitly (warehouse 'X', aperture)
    }
    if (!p.bits[d]) return PCL_ERR_INVALID;
  }
  for (int k = 0; k < n_chars; ++k) {
    p.chars[k] = chars[k];
    p.sprite_of[k] = -1; p.drape_of[k] = -1;
    for (int s = 0; s < sp.n_sprites; ++s) if (sp.sprite_char[s] == chars[k]) p.sprite_of[k] = (int8_t)s;
    for (int d = 0; d < sp.n_drapes; ++d) if (sp.drape_char[d] == chars[k]) p.drape_of[k] = (int8_t)d;
  }
  return launched(h, pcl::launch_layers(p, (cudaStream_t)stream), "launch_layers");
}

namespace {
// cropping.py:362-391: what a ScrollingCropper / FixedCropper accepts.
int crop_spec_ok(const pcl_handle* h, const pcl_crop_spec* crop) {
  if (crop->rows <= 0 || crop->cols <= 0) return PCL_ERR_INVALID;
  if (crop->track[0] == 0 && crop->sprite_index >= h->spec.n_sprites) return PCL_ERR_INVALID;
  if (crop->sprite_index >= 0 &&
      (2 * crop->margin_rows >= crop->rows || 2 * crop->margin_cols >= crop->cols))
    return PCL_ERR_INVALID;                                  // cropping.py:374-380
  if (crop->pad_char < 0 && (crop->rows > h->spec.rows || crop->cols > h->spec.cols))
    return PCL_ERR_INVALID;                                  // cropping.py:384-391
  return PCL_OK;
}
}  // namespace

int pcl_attach_cropper(pcl_handle* h, const pcl_crop_spec* crop, uint8_t* d_crop,
                       int32_t* d_crop_state) {
  if (!h) return PCL_ERR_INVALID;
  if (!h->bound) return PCL_ERR_UNBOUND;
  if (!crop) {                                               // detach
    h->base.has_cropper = 0;
    return PCL_OK;
  }
  if (!d_crop) return PCL_ERR_INVALID;
  if (h->spec.program != PCL_PROG_SCROLLY_MAZE) return PCL_ERR_UNSUPPORTED;
  const int ok = crop_spec_ok(h, crop);
  if (ok != PCL_OK) return ok;
  if ((int64_t)crop->rows * crop->cols >= 65536) return PCL_ERR_UNSUPPORTED;
  for (int i = 0; i < PCL_MAX_TRACK; ++i) {
    if (crop->track[i] < 0) return PCL_ERR_UNSUPPORTED;      // drape medians need scratch memory
    if (crop->track[i] > h->spec.n_sprites) return PCL_ERR_INVALID;
  }
  pcl::CropParams& c = h->base.cropper;
  memset(&c, 0, sizeof(c));
  c.B = h->batch; c.H = h->spec.rows; c.W = h->spec.cols; c.pitch = h->spec.pitch;
  c.S = h->spec.n_sprites; c.crop = *crop;
  c.sprites = h->st.d_sprites; c.plot = h->st.d_plot; c.out = d_crop; c.state = d_crop_state;
  c.cols_recip = crop->cols > 1 ? (uint32_t)(0x100000000ull / (uint32_t)crop->cols) + 1u : 0u;
  h->base.has_cropper = 1;
  return PCL_OK;
}

int pcl_crop(pcl_handle* h, const pcl_crop_spec* crop, const uint8_t* d_board, uint8_t* d_crop,
             int32_t* d_crop_state, void* stream) {
  return pcl_crop_tracking(h, crop, d_board, d_crop, d_crop_state, nullptr, stream);
}

int pcl_crop_tracking(pcl_handle* h, const pcl_crop_spec* crop, const uint8_t* d_board,
                      uint8_t* d_crop, int32_t* d_crop_state,
                      const uint8_t* const* d_curtains, void* stream) {
  Range nvtx_range("pcl_crop (ScrollingCropper.crop)");
  if (!h || !crop || !d_board || !d_crop) return PCL_ERR_INVALID;
  if (!h->bound) return PCL_ERR_UNBOUND;
  if (crop->rows <= 0 || crop->cols <= 0) return PCL_ERR_INVALID;
  // sprite_index names the tracked sprite only when no priority list is given (a
  // cropper may track a drape in a game without sprites).
  if (crop->track[0] == 0 && crop->sprite_index >= h->spec.n_sprites) return PCL_ERR_INVALID;
  if (crop->sprite_index >= 0 &&
      (2 * crop->margin_rows >= crop->rows || 2 * crop->margin_cols >= crop->cols))
    return PCL_ERR_INVALID;                                  // cropping.py:374-380
  if (crop->pad_char < 0 && (crop->rows > h->spec.rows || crop->cols > h->spec.cols))
    return PCL_ERR_INVALID;                                  // cropping.py:384-391
  pcl::CropParams p;
  memset(&p, 0, sizeof(p));
  p.B = h->batch; p.H = h->spec.rows; p.W = h->spec.cols; p.pitch = h->spec.pitch;
  p.S = h->spec.n_sprites; p.crop = *crop;
  p.sprites = h->st.d_sprites; p.plot = h->st.d_plot; p.board = d_board; p.out = d_crop;
  p.state = d_crop_state;
  for (int i = 0; i < PCL_MAX_TRACK; ++i) {
    const int code = crop->track[i];
    if (code == 0) break;
    if (crop->sprite_index < 0) return PCL_ERR_INVALID;      // a FixedCropper tracks nothing
    if (code > 0) {
      if (code - 1 >= h->spec.n_sprites) return PCL_ERR_INVALID;
    } else {
      if (-code - 1 >= h->spec.n_drapes || !d_curtains || !d_curtains[i]) return PCL_ERR_INVALID;
      if (h->spec.rows > 128 || h->spec.cols > 128) return PCL_ERR_UNSUPPORTED;
      p.curtains[i] = d_curtains[i];
    }
  }
  return launched(h, pcl::launch_crop(p, (cudaStream_t)stream), "launch_crop");
}

int pcl_crop_handoff(pcl_handle* h, const pcl_crop_spec* crop, const uint8_t* d_board,
                     int32_t* d_crop_state, const pcl_outputs* out, const pcl_handoff* x,
                     void* stream) {
  Range nvtx_range("pcl_crop_handoff");
  if (!h || !crop || !d_board || !out || !x) return PCL_ERR_INVALID;
  if (!h->bound) return PCL_ERR_UNBOUND;
  if (!out->d_reward || !out->d_has_reward || !out->d_discount || !out->d_done)
    return PCL_ERR_INVALID;
  if (crop->rows <= 0 || crop->cols <= 0 || crop->sprite_index >= h->spec.n_sprites)
    return PCL_ERR_INVALID;
  for (int i = 0; i < PCL_MAX_TRACK; ++i)
    if (crop->track[i] < 0) return PCL_ERR_UNSUPPORTED;      // drape tracking: pcl_crop_tracking
  if (crop->sprite_index >= 0 &&
      (2 * crop->margin_rows >= crop->rows || 2 * crop->margin_cols >= crop->cols))
    return PCL_ERR_INVALID;
  if (crop->pad_char < 0 && (crop->rows > h->spec.rows || crop->cols > h->spec.cols))
    return PCL_ERR_INVALID;
  const int view = crop->rows * crop->cols;
  if (x->n_peers < 1 || x->n_peers > PCL_MAX_PEERS || x->rank < 0 || x->rank >= x->n_peers)
    return PCL_ERR_INVALID;
  if ((x->record_bytes & 15) || x->record_bytes < PCL_HANDOFF_RECORD_BYTES(view) ||
      x->record_bytes > 256) return PCL_ERR_INVALID;
  if (!x->d_local || x->first_row < 0 || x->first_row + h->batch > x->rows) return PCL_ERR_INVALID;
  pcl::CropParams p;
  memset(&p, 0, sizeof(p));
  p.B = h->batch; p.H = h->spec.rows; p.W = h->spec.cols; p.pitch = h->spec.pitch;
  p.S = h->spec.n_sprites; p.crop = *crop;
  p.sprites = h->st.d_sprites; p.plot = h->st.d_plot; p.board = d_board; p.out = nullptr;
  p.state = d_crop_state;
  pcl::HandoffParams q;
  memset(&q, 0, sizeof(q));
  q.n_peers = x->n_peers; q.rank = x->rank; q.record_bytes = x->record_bytes;
  q.rows = x->rows; q.first_row = x->first_row;
  for (int i = 0; i < x->n_peers; ++i) {
    if (!x->d_peer_base[i] || !x->d_peer_flags[i]) return PCL_ERR_INVALID;
    q.peer_base[i] = x->d_peer_base[i]; q.peer_flags[i] = x->d_peer_flags[i];
  }
  q.multicast = x->d_multicast; q.local = x->d_local; q.out = *out;
  q.n_bufs = x->n_bufs == 0 ? 2 : x->n_bufs;
  if (x->mode & ~(PCL_HANDOFF_LAG | PCL_HANDOFF_SIGNAL_KERNEL)) return PCL_ERR_INVALID;
  q.lag = (x->mode & PCL_HANDOFF_LAG) ? 1 : 0;
  q.signal_kernel = (x->mode & PCL_HANDOFF_SIGNAL_KERNEL) ? 1 : 0;
  if (q.n_bufs < 2 || q.n_bufs > 8 || (q.lag == 1 && q.n_bufs < 3)) return PCL_ERR_INVALID;
  const int r = launched(h, pcl::launch_crop_handoff(p, q, (cudaStream_t)stream), "launch_crop_handoff");
  if (r == PCL_OK && q.signal_kernel) h->launches += 1;      // the one-warp publish kernel
  return r;
}

int pcl_pack_handoff(pcl_handle* h, const uint8_t* d_view, int32_t view_bytes,
                     const pcl_outputs* out, uint8_t* d_packed, void* stream) {
  if (!h || !d_view || !out || !d_packed || view_bytes <= 0) return PCL_ERR_INVALID;
  if (!out->d_reward || !out->d_has_reward || !out->d_discount || !out->d_done)
    return PCL_ERR_INVALID;
  pcl::PackParams p;
  memset(&p, 0, sizeof(p));
  p.B = h->batch; p.view_bytes = view_bytes;
  p.record_bytes = PCL_HANDOFF_RECORD_BYTES(view_bytes);
  p.view = d_view; p.out = *out; p.packed = d_packed;
  return launched(h, pcl::launch_pack_handoff(p, (cudaStream_t)stream), "launch_pack_handoff");
}

int pcl_pack_handoff_peers(pcl_handle* h, const uint8_t* d_view, int32_t view_bytes,
                           const pcl_outputs* out, uint8_t* const* d_peer_bases,
                           int32_t n_peers, int64_t first_row, void* stream) {
  if (!h || !d_view || !out || !d_peer_bases || view_bytes <= 0 || first_row < 0)
    return PCL_ERR_INVALID;
  if (n_peers < 1 || n_peers > PCL_MAX_PEERS) return PCL_ERR_INVALID;
  if (!out->d_reward || !out->d_has_reward || !out->d_discount || !out->d_done)
    return PCL_ERR_INVALID;
  pcl::PackParams p;
  memset(&p, 0, sizeof(p));
  p.B = h->batch; p.view_bytes = view_bytes;
  p.record_bytes = PCL_HANDOFF_RECORD_BYTES(view_bytes);
  p.view = d_view; p.out = *out;
  p.n_peers = n_peers; p.first_row = first_row;
  for (int i = 0; i < n_peers; ++i) {
    if (!d_peer_bases[i]) return PCL_ERR_INVALID;
    p.peers[i] = d_peer_bases[i];
  }
  return launched(h, pcl::launch_pack_handoff(p, (cudaStream_t)stream), "launch_pack_handoff");
}

int pcl_observe(pcl_handle* h, const pcl_observe_spec* spec, const void* d_table,
                const uint8_t* d_valid, const uint8_t* d_board, void* d_out,
                int32_t* d_unknown, void* stream) {
  Range nvtx_range("pcl_observe");
  if (!h || !spec || !d_table || !d_board || !d_out) return PCL_ERR_INVALID;
  if (spec->depth < 1 || spec->depth > 32 || spec->dtype < 0 || spec->dtype > 4)
    return PCL_ERR_INVALID;
  pcl::ObserveParams p;
  memset(&p, 0, sizeof(p));
  p.B = h->batch; p.H = h->spec.rows; p.W = h->spec.cols; p.pitch = h->spec.pitch;
  p.depth = spec->depth; p.dtype = spec->dtype;
  p.words = spec->dtype >= 3 ? 2 : 1;
  p.stride_b = spec->stride_b * p.words; p.stride_d = spec->stride_d * p.words;
  p.stride_r = spec->stride_r * p.words; p.stride_c = spec->stride_c * p.words;
  p.table = d_table; p.valid = d_valid; p.board = d_board; p.out = d_out;
  p.unknown = d_unknown;
  return launched(h, pcl::launch_observe(p, (cudaStream_t)stream), "launch_observe");
}

int pcl_error_codes(pcl_handle* h, int32_t* d_out, void* stream) {
  if (!h || !d_out) return PCL_ERR_INVALID;
  if (!h->bound) return PCL_ERR_UNBOUND;
  gather_errors<<<(h->batch + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->st.d_plot, d_out,
                                                                           h->batch);
  return launched(h, cudaGetLastError(), "gather_errors");
}

int pcl_launch_count(pcl_handle* h, int64_t* out) {
  if (!h || !out) return PCL_ERR_INVALID;
  *out = h->launches;
  return PCL_OK;
}

}  // extern "C"
