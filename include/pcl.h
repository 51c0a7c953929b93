/*
 * pcl.h — C ABI of the B200 batched gridworld step engine (libpcl.so).
 *
 * pycolab has no FFI: its "plugin interface" for the per-step hot path is the
 * Python object API  Engine.its_showtime() / Engine.play(actions)  returning
 * (Observation(board, layers), reward, discount)  (reference
 * pycolab/engine.py:520-639).  This header is what a native replacement of
 * that path exports; INTEGRATION.md shows the ctypes binding a pycolab
 * maintainer would add.  Conventions (SURVEY.md §8b):
 *
 *   - plain C, no C++/torch types; every pointer named d_* is a DEVICE
 *     pointer, h_* a HOST pointer; buffers are owned by the caller, the
 *     library never frees them;
 *   - every entry point returns 0 (PCL_OK) or a negative pcl_status and never
 *     throws; per-environment run-time faults (the reference's RuntimeError /
 *     scrolling.Error cases) are latched in a per-env error word readable
 *     with pcl_error_codes();
 *   - every launch takes the cudaStream_t (as void*) to enqueue on; nothing
 *     synchronises except the *_host entry points;
 *   - re-entrant per handle, no global state.
 *
 * Batched-state model: B independent environments ("envs"), each the
 * equivalent of one reference Engine, live as a struct-of-arrays in HBM.
 * One warp advances one env per launch.
 */
#ifndef PCL_H_
#define PCL_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCL_ABI_VERSION 2

#define PCL_MAX_SPRITES 16
#define PCL_MAX_DRAPES 8
#define PCL_SPRITE_WORDS 8   /* int32 words per sprite record */
#define PCL_DRAPE_WORDS 8    /* int32 words per drape record  */
#define PCL_PLOT_WORDS 16    /* int32 words per env plot record */
#define PCL_MT_WORDS 625     /* MT19937: 624 state words + position */
#define PCL_MAX_SCROLL_GROUPS 4 /* scrolling groups of one game (protocols/scrolling.py:198-241) */
#define PCL_GROUP_WORDS 4    /* int32 words per scrolling-group record */

typedef enum pcl_status {
  PCL_OK = 0,
  PCL_ERR_INVALID = -1,      /* bad argument / malformed spec (ValueError)   */
  PCL_ERR_UNSUPPORTED = -2,  /* spec is valid pycolab but not lowered        */
  PCL_ERR_CUDA = -3,         /* a CUDA runtime call failed                   */
  PCL_ERR_UNBOUND = -4,      /* pcl_bind_state has not been called           */
  PCL_ERR_NOMEM = -5
} pcl_status;

/* Per-env latched error bits (pcl_error_codes).  Each mirrors an exception
 * the reference would raise inside Engine.play(). */
#define PCL_ENV_ERR_ORDER_MISMATCH   0x1  /* sprites.py:449-454, drapes.py:525-530 */
#define PCL_ENV_ERR_SECOND_ORDER     0x2  /* scrolling.py:518-521 */
#define PCL_ENV_ERR_EMPTY_CHOICE     0x4  /* np.random.choice([]) in marauders :253 */
#define PCL_ENV_ERR_INDEX            0x8  /* NumPy IndexError (board look-up off the array) */
#define PCL_ENV_ERR_BAD_Z            0x10 /* change_z_order names a missing entity, engine.py:802-812 */

/* Which game program advances the envs.  One fused kernel per program; the
 * host "lowering" recognises the reference's entity classes and picks one. */
typedef enum pcl_program {
  PCL_PROG_NONE = 0,         /* no step program: pcl_render / pcl_crop only        */
  PCL_PROG_SCROLLY_MAZE = 1, /* examples/scrolly_maze.py:212-364               */
  PCL_PROG_WAREHOUSE = 2,    /* examples/warehouse_manager.py:139-295          */
  PCL_PROG_MARAUDERS = 3,    /* examples/extraterrestrial_marauders.py:91-256  */
  PCL_PROG_FIXTURE = 4,      /* tests/test_things.py TestMazeWalker/TestScrolly */
  PCL_PROG_BETTER_SCROLLY = 5, /* examples/better_scrolly_maze.py:209-324       */
  PCL_PROG_CLASSICS = 6,     /* one-walker games: examples/classics/{four_rooms,cliff_walk,
                                chain_walk}.py, examples/fluvial_natation.py */
  PCL_PROG_APERTURE = 7,     /* examples/aperture.py:118-196; the drape record's AUX0 / AUX1 hold
                                the two aperture cells (row << 16 | col, -1 = none) */
  PCL_PROG_HELLO = 9,        /* examples/hello_world.py:58-118: plain Sprites (aux0 = direction set)
                                + one rolling Drape (record AUX0 / AUX1 = row / column shift of the
                                reset curtain); program_arg[0..n) = the z-order chars */
  PCL_PROG_APPREHEND = 10,   /* examples/apprehend.py:56-131: sprites 'P' (confined catcher) and 'b' (falling
                                ball); the ball's AUX0 / AUX1 hold its float64 slope (bits lo / hi), plot
                                AUX0 / AUX1 its x accumulator; with pcl_state.d_rng bound (the words of
                                Python's random.Random(seed).getstate()) the slope is drawn on the device at
                                every (re)start as random.uniform does, else taken from the reset template */
  PCL_PROG_SHOCKWAVE = 11,   /* examples/shockwave.py:91-197: sprite 'P', drapes '@' (curtain bit-packed in
                                d_bits[0], record AUX0 = impact cell index, AUX1 = steps since impact), ' '
                                and '^' (static, d_bits_init[1..2]); program_arg[0] = ring width; d_rng =
                                NumPy RandomState words (np.random.randint picks the impact cell) */
  PCL_PROG_BOX_WORLD = 12,   /* examples/research/box_world/box_world.py:127-271: one MazeWalker (the
                                player, '.') and up to 41 key / lock / gem drapes, held together as
                                ONE byte plane in d_bits[0] / d_bits_init[0] (u8 [*, rows, pitch],
                                bits_words = pitch / 4): byte = the drape character covering the
                                cell, 0 = none, bit 7 set on distractor lock cells; cell (0, 0) =
                                the key held.  n_drapes = 0.  Sprite AUX0 = move actions taken,
                                AUX1 = max_num_steps.  Boards up to 32 x 32 with '#' all round.
                                Level rotation: program_arg[1] = stride (0 = off), program_arg[2]
                                = number of levels; an AUTO-reset sets d_level[env] = (d_level[env]
                                + stride) % levels before restoring the templates (pcl_reset
                                restarts the same level) */
  PCL_PROG_ORDEAL = 8        /* examples/ordeal.py:74-266: program_arg[0] = PCL_ORDEAL_* chapter;
                                plot words AUX0 has_sword, AUX1 last_position (row << 16 | col,
                                -1 unset), AUX2 next_chapter chosen on the device, AUX3 prior chapter */
} pcl_program;

/* PCL_PROG_ORDEAL chapters (storytelling.Story keys of ordeal.py:94-97); AUX2 holds
 * PCL_ORDEAL_NEXT_UNSET until an entity names the next chapter, PCL_ORDEAL_NEXT_NONE for
 * `next_chapter = None`. */
enum { PCL_ORDEAL_NEXT_UNSET = -1, PCL_ORDEAL_NEXT_NONE = 0,
       PCL_ORDEAL_CASTLE = 1, PCL_ORDEAL_CAVERN = 2, PCL_ORDEAL_KANSAS = 3 };

/* PCL_PROG_CLASSICS: pcl_spec.program_arg[0] selects the rule set; the games
 * pay float rewards (1.0, -1.0, -100.0, 100.0) which d_reward carries as the
 * equal int32 value. */
enum { PCL_CLASSIC_FOUR_ROOMS = 0, /* four_rooms.py:52-80; program_arg[1..2] = goal cell (4, 3) */
       PCL_CLASSIC_CLIFF_WALK = 1, /* cliff_walk.py:46-86 */
       PCL_CLASSIC_CHAIN_WALK = 2, /* chain_walk.py:44-73 */
       PCL_CLASSIC_FLUVIAL = 3     /* examples/fluvial_natation.py:61-110 (int rewards); program_arg[1..2] =
                                      first / end row of the flowing backdrop band (1, 4); the
                                      rotation count is plot word PCL_P_AUX0 */ };

/* Plot directives as action words of PCL_PROG_FIXTURE (plot.py:136-260). */
#define PCL_FIXTURE_DIRECTIVES 4
enum { PCL_DIR_NONE = 0,
       PCL_DIR_ADD_REWARD = 1,        /* arg = int32 reward (plot.py:201-214) */
       PCL_DIR_TERMINATE = 2,         /* arg = f32 bits of the discount in [0, 1] (plot.py:176-199) */
       PCL_DIR_DEFAULT_DISCOUNT = 3,  /* arg = f32 bits (plot.py:247-260; upstream resets the default
                                         to 1.0 after every step, plot.py:345-356) */
       PCL_DIR_Z_ORDER = 4 };         /* arg = move_this | in_front_of << 8, 0 = None (plot.py:136-174) */

/* Motion codes (prefab_parts/sprites.py:140-150). */
enum { PCL_M_N = 0, PCL_M_NE, PCL_M_E, PCL_M_SE, PCL_M_S, PCL_M_SW, PCL_M_W,
       PCL_M_NW, PCL_M_STAY, PCL_M_NONE = -1 };

/* Action value meaning "actions=None" (the its_showtime() frame,
 * engine.py:581). */
#define PCL_ACTION_NONE (-1)

/* Sprite record layout, int32[PCL_SPRITE_WORDS] (things.py:339-391,
 * sprites.py:153-205). */
enum { PCL_S_ROW = 0, PCL_S_COL, PCL_S_VROW, PCL_S_VCOL,
       PCL_S_FLAGS,          /* bit0 visible; bits1-2 prior_visible: 0 None, 1 False, 2 True */
       PCL_S_AUX0,           /* program-specific (e.g. patroller heading; permit mask)      */
       PCL_S_AUX1,           /* program-specific (e.g. permit frame)                        */
       PCL_S_AUX2 };
/* Drape record layout, int32[PCL_DRAPE_WORDS] (drapes.py:293-376). */
enum { PCL_D_CORNER_R = 0, PCL_D_CORNER_C, PCL_D_PRE_R, PCL_D_PRE_C,
       PCL_D_LAST_FRAME,     /* _last_maybe_move_frame; INT32_MIN = -inf */
       PCL_D_AUX0, PCL_D_AUX1, PCL_D_AUX2 };
/* Plot record layout, int32[PCL_PLOT_WORDS] (plot.py:69-104,
 * protocols/scrolling.py:198-241). */
enum { PCL_P_FRAME = 0, PCL_P_GAME_OVER, PCL_P_ERROR, PCL_P_EPISODES,
       PCL_P_ORDER_R, PCL_P_ORDER_C, PCL_P_ORDER_FRAME, PCL_P_EGO_MASK,
       PCL_P_AUX0, PCL_P_AUX1, PCL_P_AUX2, PCL_P_AUX3,
       PCL_P_CROP_R, PCL_P_CROP_C, PCL_P_CROP_INIT, PCL_P_RESERVED };

/* Scrolling-group record layout, int32[PCL_GROUP_WORDS]: the per-group part of the
 * blackboard of protocols/scrolling.py:198-241.  Group 0 lives in the plot record
 * (PCL_P_ORDER_R .. PCL_P_EGO_MASK); groups 1.. in pcl_state.d_groups. */
enum { PCL_G_ORDER_R = 0, PCL_G_ORDER_C, PCL_G_ORDER_FRAME, PCL_G_EGO_MASK };

/* Static description of one game (what Engine's set-up API collected:
 * engine.py:248-518).  All envs of a handle share it. */
typedef struct pcl_spec {
  int32_t abi_version;           /* PCL_ABI_VERSION */
  int32_t program;               /* pcl_program */
  int32_t rows, cols;            /* board H x W (engine.py:202-203) */
  int32_t pitch;                 /* bytes per board row in HBM, multiple of 16, >= cols */
  int32_t n_sprites, n_drapes;
  int32_t auto_reset;            /* 1: an env that is game-over is rebuilt by the next step */
  int32_t pattern_rows, pattern_cols; /* Scrolly whole_pattern shape (drapes.py:338-343) */
  int32_t pattern_words;         /* uint32 words per bit-packed pattern row: >= ceil(cols/32) + 2 (zero padded) */
  int32_t bits_words;            /* uint32 words per bit-packed board-sized row */
  uint8_t sprite_char[PCL_MAX_SPRITES];
  uint8_t drape_char[PCL_MAX_DRAPES];
  uint32_t impassable[PCL_MAX_SPRITES][4]; /* 128-bit ASCII set (sprites.py:190) */
  int32_t sprite_confined[PCL_MAX_SPRITES];
  int32_t sprite_egocentric[PCL_MAX_SPRITES];
  int32_t margins[PCL_MAX_DRAPES][2];      /* Scrolly scroll_margins; -1,-1 = None */
  uint8_t z_order[PCL_MAX_SPRITES + PCL_MAX_DRAPES]; /* initial z-order, chars */
  int32_t n_groups;
  int32_t group_len[PCL_MAX_SPRITES + PCL_MAX_DRAPES];
  uint8_t group_chars[PCL_MAX_SPRITES + PCL_MAX_DRAPES]; /* update order, concatenated */
  int32_t drape_kind[PCL_MAX_DRAPES];      /* 0 = plain bool curtain (d_bits), 1 = Scrolly (d_pattern) */
  int32_t program_arg[8];                  /* per-program constants (see pcl_program); else 0 */
  /* Scrolling groups (`scrolling_group` of MazeWalker / Scrolly, sprites.py:176,
   * drapes.py:309): index of each entity's group, 0 .. n_scroll_groups - 1.  Only
   * PCL_PROG_FIXTURE accepts more than one group; 0 groups means 1. */
  int32_t n_scroll_groups;
  int32_t sprite_group[PCL_MAX_SPRITES];
  int32_t drape_group[PCL_MAX_DRAPES];
} pcl_spec;

/* Device buffers of one handle (all caller-owned).  A "*_bstride" is the
 * distance between consecutive envs in ELEMENTS of that array; 0 means all
 * envs share one copy (legal only for arrays the step never writes). */
typedef struct pcl_state {
  /* static level data */
  const uint8_t* d_backdrop;   int64_t backdrop_bstride;       /* u8 [*, rows, pitch] */
  /* Scrolly patterns, bit-packed: u32 [*, pattern_rows, pattern_words], cell c
   * of a row is bit (c & 31) of word (c >> 5). */
  uint32_t* d_pattern[PCL_MAX_DRAPES];  int64_t pattern_bstride[PCL_MAX_DRAPES];
  const uint32_t* d_pattern_init[PCL_MAX_DRAPES]; int64_t pattern_init_bstride[PCL_MAX_DRAPES];
  /* board-sized bit-packed curtains for non-Scrolly drapes: u32 [*, rows, bits_words] */
  uint32_t* d_bits[PCL_MAX_DRAPES];     int64_t bits_bstride[PCL_MAX_DRAPES];
  const uint32_t* d_bits_init[PCL_MAX_DRAPES]; int64_t bits_init_bstride[PCL_MAX_DRAPES];
  /* per-env registers and their reset templates */
  int32_t* d_sprites;  const int32_t* d_sprites_init; int64_t sprites_init_bstride; /* [B, S, 8] */
  int32_t* d_drapes;   const int32_t* d_drapes_init;  int64_t drapes_init_bstride;  /* [B, D, 8] */
  int32_t* d_plot;     const int32_t* d_plot_init;    int64_t plot_init_bstride;    /* [B, 16]   */
  uint32_t* d_rng;     /* MT19937 per env, u32 [B, PCL_MT_WORDS]; NULL if unused */
  /* per-env z-order (chars, back to front) for programs whose entities issue
   * Plot.change_z_order (engine.py:796-835): u8 [B, n_sprites + n_drapes]; NULL = spec z_order */
  uint8_t* d_z_order;  const uint8_t* d_z_order_init; int64_t z_order_init_bstride;
  /* Scrolling groups 1 .. n_scroll_groups - 1 (group 0 is in the plot record):
   * i32 [B, PCL_MAX_SCROLL_GROUPS, PCL_GROUP_WORDS], slot 0 unused; NULL when the
   * game has a single group. */
  int32_t* d_groups;   const int32_t* d_groups_init;  int64_t groups_init_bstride;
  /* Level sharing: envs that play the same level need only one copy of its
   * static data.  When d_level (i32 [B]) is non-NULL, every array the step never
   * writes — d_backdrop, read-only patterns, every *_init template — is indexed
   * by d_level[env] instead of env (the *_bstride is then the per-LEVEL stride);
   * mutable arrays stay env-indexed.  NULL = env-indexed (or bstride 0).  The
   * library writes it only for PCL_PROG_BOX_WORLD with level rotation on. */
  int32_t* d_level;
} pcl_state;

/* Per-step outputs = the (observation, reward, discount) triple of
 * Engine.play() (engine.py:639) plus Engine.game_over (engine.py:657). */
typedef struct pcl_outputs {
  uint8_t* d_board;       /* u8 [B, rows, pitch]; Observation.board.  PCL_PROG_FIXTURE reads the
                             board of the LAST render back from here at the next step (its
                             entities may test any character, engine.py:725-735): pass the same
                             d_board to consecutive steps of a handle running that program. */
  int32_t* d_reward;      /* i32 [B]; summed reward (plot.py:201-214), 0 if none */
  uint8_t* d_has_reward;  /* u8 [B]; 0 = reference returned reward None */
  float*   d_discount;    /* f32 [B]; 1.0 running / 0.0 terminated unless a directive said otherwise
                             (plot.py:104,176-199,247-260) */
  uint8_t* d_done;        /* u8 [B]; Engine.game_over after this step */
} pcl_outputs;

typedef struct pcl_handle pcl_handle;

/* Validate `spec`, allocate the handle.  Replaces Engine.__init__ + set-up
 * bookkeeping (engine.py:191-246). */
int pcl_create(const pcl_spec* spec, int batch, int device, pcl_handle** out);
int pcl_destroy(pcl_handle* h);

/* Attach the caller's device buffers. */
int pcl_bind_state(pcl_handle* h, const pcl_state* state);

/* Engine.its_showtime() (engine.py:520-581) for every env whose d_env_mask
 * byte is non-zero (NULL = all): restore the reset templates, then run the
 * actions=None frame.  Envs not selected are left untouched. */
int pcl_reset(pcl_handle* h, const uint8_t* d_env_mask, const pcl_outputs* out,
              void* stream);

/* Engine.play(actions) (engine.py:583-639) for all envs in lockstep: one fused
 * kernel = _update_and_render + _apply_and_clear_plot.  d_actions is
 * i32 [B, actions_per_env]: actions_per_env = 1 for the example games;
 * PCL_PROG_FIXTURE takes n_sprites + n_drapes + 2 * PCL_FIXTURE_DIRECTIVES words per
 * env: one motion code per entity in update order, then PCL_FIXTURE_DIRECTIVES
 * (opcode, argument) pairs — the Plot directives the entities issued this step, in
 * call order (the last discount-setting call wins, as upstream). */
int pcl_step(pcl_handle* h, const int32_t* d_actions, const pcl_outputs* out,
             void* stream);

/* T consecutive pcl_step()s with d_actions i32 [T, B, actions_per_env]; the
 * outputs hold the last step's values. */
int pcl_run(pcl_handle* h, const int32_t* d_actions, int steps,
            const pcl_outputs* out, void* stream);

/* `steps` pcl_step()s issued from one C call over several handles in rotation:
 * step t advances handles[t % n_handles] with d_actions[t] (HOST array of `steps`
 * device pointers, each i32 [B, actions_per_env] of that handle) into
 * outs[t % n_handles].  The batched stand-in for a driver looping over many
 * Engines (one reference Engine per env, engine.py:583); nothing but kernel
 * launches sits between the steps, so the sequence can also be captured into a
 * CUDA graph on `stream`. */
int pcl_run_many(pcl_handle* const* handles, int n_handles, const int32_t* const* d_actions,
                 const pcl_outputs* const* outs, int steps, void* stream);

/* Host-buffer form of pcl_step: copies h_actions to the device, steps, copies
 * the outputs back into the h_* buffers (any may be NULL = skip) and
 * synchronises the stream.  `out` names the device staging buffers. */
int pcl_step_host(pcl_handle* h, const int32_t* h_actions, int32_t* d_actions,
                  const pcl_outputs* out, uint8_t* h_board, int32_t* h_reward,
                  uint8_t* h_has_reward, float* h_discount, uint8_t* h_done,
                  void* stream);

/* Pipelined form of pcl_step_host.  Enqueues H2D(actions) and the step on
 * `stream`, then the D2H of the requested outputs on a handle-owned copy stream
 * behind it, and returns WITHOUT synchronising: the copies of this step overlap
 * whatever is enqueued on `stream` next (another handle's step, or this handle's
 * next step once its outputs were read).  `slot` (0 .. PCL_HOST_SLOTS - 1) names
 * the completion event; pcl_host_wait(h, slot) blocks until the h_* buffers of
 * that call are valid.  Until then the caller must leave h_actions and the h_*
 * buffers alone, and must not call the synchronous step entry points on `h`.
 * With `crop` non-NULL the step is followed by pcl_crop(crop, d_crop, d_crop_state)
 * and h_view receives the crops u8 [B, crop rows, crop cols] instead of the
 * boards u8 [B, rows, pitch] — only the view the agent consumes crosses PCIe
 * (cropping.py:393-426 applied before the hand-off). */
#define PCL_HOST_SLOTS 8
struct pcl_crop_spec;
int pcl_step_host_async(pcl_handle* h, const int32_t* h_actions, int32_t* d_actions,
                        const pcl_outputs* out, const struct pcl_crop_spec* crop,
                        uint8_t* d_crop, int32_t* d_crop_state, uint8_t* h_view,
                        int32_t* h_reward, uint8_t* h_has_reward, float* h_discount,
                        uint8_t* h_done, int slot, void* stream);
int pcl_host_wait(pcl_handle* h, int slot);

/* Stand-alone renderer = Engine._render() + BaseObservationRenderer
 * (engine.py:737-759, rendering.py:98-179) over reference-layout inputs:
 * u8 backdrop [*, rows, pitch], byte curtains u8 [B, n_drapes, rows, pitch],
 * sprite records, per-env z-order u8 [B, n_sprites + n_drapes] of chars. */
int pcl_render(pcl_handle* h, const uint8_t* d_backdrop, int64_t backdrop_bstride,
               const uint8_t* d_curtains, const int32_t* d_sprites,
               const uint8_t* d_z_order, uint8_t* d_board, void* stream);

/* Byte-per-cell view of drape `drape_index`'s current curtain (Drape.curtain,
 * things.py:213-217): u8 [B, rows, pitch]. */
int pcl_export_curtain(pcl_handle* h, int drape_index, uint8_t* d_out, void* stream);

/* Layers of BaseUnoccludedObservationRenderer (rendering.py:187-301, selected by
 * Engine(occlusion_in_layers=False), engine.py:564-570) for the whole batch: plane k
 * of d_out u8 [B, n_chars, rows, pitch] is 1 wherever the owner of chars[k] places it,
 * occluded or not — the backdrop where it holds that character, a drape's whole
 * curtain, a visible sprite's cell.  `chars` is a HOST array of n_chars <= 32 ASCII
 * codes.  PCL_ERR_UNSUPPORTED for programs whose drape curtain is implicit
 * (warehouse 'X', aperture). */
int pcl_layers(pcl_handle* h, const uint8_t* chars, int32_t n_chars, uint8_t* d_out,
               void* stream);

/* ScrollingCropper.crop (cropping.py:393-426): track sprite `sprite_index`,
 * update the per-env window corner and copy the crop_rows x crop_cols window of
 * d_board into d_crop u8 [B, crop_rows, crop_cols].  The corner lives in
 * d_crop_state, i32 [B, 4] = (row, col, initialised, episode) owned by the
 * caller, one array per cropper object (zero-filled at creation); a window
 * re-initialises itself when the env's episode counter moves on, as
 * ScrollingCropper.set_engine does for a new Engine (cropping.py:375-391).
 * d_crop_state == NULL selects a single built-in cropper slot in the plot record.
 * sprite_index < 0 is a FixedCropper at (offset_rows, offset_cols). */
#define PCL_MAX_TRACK 4
typedef struct pcl_crop_spec {
  int32_t rows, cols;          /* window shape */
  int32_t sprite_index;        /* entity to track (a sprite) */
  int32_t pad_char;            /* ASCII code, or -1 for None */
  int32_t margin_rows, margin_cols; /* resolved scroll margins (cropping.py:362-373) */
  int32_t offset_rows, offset_cols; /* initial_offset */
  int32_t saccade;
  int32_t track[PCL_MAX_TRACK];     /* optional priority list (pcl_crop_tracking): k > 0 = sprite
                                       k - 1, k < 0 = drape -k - 1, 0 = end; all 0 = [sprite_index] */
} pcl_crop_spec;
int pcl_crop(pcl_handle* h, const pcl_crop_spec* crop, const uint8_t* d_board,
             uint8_t* d_crop, int32_t* d_crop_state, void* stream);

/* Attach ONE cropper to the handle: every later pcl_reset / pcl_step / pcl_run then also
 * writes the cropper's view of the new board into d_crop (u8 [B, rows, cols]) from INSIDE
 * the step kernel — what pcl_crop would produce if called right after the step, without
 * the second launch.  d_crop_state as for pcl_crop (NULL = the plot record's slot).
 * crop == NULL detaches.  Step programs without the epilogue (today every program but
 * PCL_PROG_SCROLLY_MAZE) and tracking lists that name drapes return PCL_ERR_UNSUPPORTED:
 * call pcl_crop after the step instead.  The buffers must outlive the attachment;
 * pcl_bind_state detaches.  pcl_step_host_async given the SAME spec, d_crop and
 * d_crop_state does not launch the cropper a second time. */
int pcl_attach_cropper(pcl_handle* h, const pcl_crop_spec* crop, uint8_t* d_crop,
                       int32_t* d_crop_state);

/* pcl_crop for a ScrollingCropper whose `to_track` names several entities
 * (cropping.py:544-598): the window follows the FIRST entry of crop->track that is
 * visible — a sprite that is visible, or a drape whose curtain has any cell, in
 * which case the position is (median row, median column) of its cells, truncated.
 * d_curtains[i] is the curtain of the drape named by track[i] as u8 [B, rows, pitch]
 * (what pcl_export_curtain writes); entries for sprites are ignored and may be
 * NULL.  Boards up to 128 x 128 when a drape is tracked. */
int pcl_crop_tracking(pcl_handle* h, const pcl_crop_spec* crop, const uint8_t* d_board,
                      uint8_t* d_crop, int32_t* d_crop_state,
                      const uint8_t* const* d_curtains, void* stream);

/* Observation post-processors as one table look-up per cell
 * (rendering.py:304-661): out[b, d, r, c] = table[board[b, r, c]][d].
 *   ObservationCharacterRepainter: depth 1, u8 table = the character mapping;
 *   ObservationToArray:            the value mapping (scalars or depth-vectors);
 *   ObservationToFeatureArray:     f32 one-hot, table[ch][d] = (ch == layers[d]).
 * d_table is [128, depth] of `dtype`; d_valid u8 [128] marks characters the
 * mapping knows (NULL = all); a board holding an unknown character sets
 * *d_unknown (i32, may be NULL) to 1 (upstream RuntimeError, rendering.py:520-526).
 * Output strides are in ELEMENTS, so any `permute` is just a stride choice. */
typedef struct pcl_observe_spec {
  int32_t depth;
  int32_t dtype;              /* 0 uint8, 1 int32, 2 float32, 3 int64, 4 float64 */
  int64_t stride_b, stride_d, stride_r, stride_c;
} pcl_observe_spec;
int pcl_observe(pcl_handle* h, const pcl_observe_spec* spec, const void* d_table,
                const uint8_t* d_valid, const uint8_t* d_board, void* d_out,
                int32_t* d_unknown, void* stream);

/* Multi-GPU hand-off record (SURVEY.md 8e): everything one env contributes to the
 * per-step all-gather, packed so that ONE collective moves it all.
 *   d_packed u8 [B, record_bytes]; one record = view_bytes of the env's observation
 *   view (e.g. its 9x9 crop, row-major; d_view is u8 [B, view_bytes]), zero padding
 *   to a multiple of 4, then reward i32, discount f32, done u8, has_reward u8 and
 *   2 padding bytes; record_bytes = PCL_HANDOFF_RECORD_BYTES(view_bytes). */
#define PCL_HANDOFF_RECORD_BYTES(view_bytes) ((((view_bytes) + 3) & ~3) + 12)
int pcl_pack_handoff(pcl_handle* h, const uint8_t* d_view, int32_t view_bytes,
                     const pcl_outputs* out, uint8_t* d_packed, void* stream);

/* pcl_pack_handoff with the all-gather fused into the producing kernel: every
 * record is stored straight into the gather buffer of EVERY rank over NVLink
 * (peer-to-peer stores), so no collective library call sits between the step and
 * its consumers.  d_peer_bases (a HOST array of n_peers <= PCL_MAX_PEERS peer-mapped
 * device pointers, e.g. torch symmetric memory) are the bases of the ranks' gather
 * buffers u8 [rows, record_bytes]; this handle's env e lands in row first_row + e
 * of each.  The caller orders steps with a cross-GPU barrier (the records are
 * complete on every peer once this kernel has finished on every rank). */
#define PCL_MAX_PEERS 8
int pcl_pack_handoff_peers(pcl_handle* h, const uint8_t* d_view, int32_t view_bytes,
                           const pcl_outputs* out, uint8_t* const* d_peer_bases,
                           int32_t n_peers, int64_t first_row, void* stream);

/* ScrollingCropper.crop + pcl_pack_handoff_peers + the cross-GPU barrier in ONE
 * kernel (SURVEY.md 8e; cropping.py:393-426 for the view): every env's record —
 * its crop_rows x crop_cols window, zero padding to a multiple of 4, reward i32,
 * discount f32, done u8, has_reward u8, then zero padding up to `record_bytes` — is
 * stored with 16-byte stores into row first_row + env of EVERY rank's gather buffer
 * over NVLink (or once through `d_multicast`, the NVLS multicast mapping of those
 * buffers).  The last thread block to finish publishes this rank's step count in
 * every peer's flag array and waits until every peer has published the same count
 * here: when the kernel retires, half (step & 1) of the LOCAL gather buffer holds
 * all ranks' records of this step.  No collective call and no separate barrier
 * kernel; the step count lives in device memory (`d_local`), so the launch can be
 * captured in a CUDA graph.  Every rank must make the same sequence of calls.
 *   gather buffer of a rank: u8 [n_bufs, rows, record_bytes]  (parts alternate by step)
 *   flag array of a rank:    u32 [PCL_MAX_PEERS], zero-initialised; word s = steps
 *                            whose records from rank s have landed here
 *   d_local:                 u32 [2] zero-initialised device memory of this rank
 * record_bytes: multiple of 16, >= PCL_HANDOFF_RECORD_BYTES(crop rows * cols), <= 256. */
#define PCL_HANDOFF_LAG 1
#define PCL_HANDOFF_SIGNAL_KERNEL 2
typedef struct pcl_handoff {
  int32_t n_peers, rank;
  int32_t record_bytes;
  int64_t rows, first_row;
  uint8_t* d_peer_base[PCL_MAX_PEERS];   /* peer-mapped: every rank's gather buffer */
  uint32_t* d_peer_flags[PCL_MAX_PEERS]; /* peer-mapped: every rank's flag array   */
  uint8_t* d_multicast;                  /* multicast mapping of the gather buffers, or NULL */
  uint32_t* d_local;
  int32_t n_bufs;   /* parts of a gather buffer that alternate by step: 0 or 2 = two halves */
  int32_t mode;     /* bit flags:
                     * PCL_HANDOFF_LAG (1), split phase: signal this step but only wait for the
                     *   PREVIOUS one, so the cross-GPU wait leaves the critical path: when the call
                     *   for step s retires, part (s - 1) % n_bufs holds every rank's records of step
                     *   s - 1.  Needs n_bufs >= 3 (a peer one step ahead writes part (s + 1) % n_bufs
                     *   while part (s - 1) % n_bufs is being read); the last step is completed by any
                     *   host-level barrier after the stream has drained.
                     * PCL_HANDOFF_SIGNAL_KERNEL (2): the records kernel neither fences nor counts
                     *   blocks; a second, one-warp kernel behind it (the kernel boundary completes
                     *   the peer stores) publishes the flags and waits.  Measured faster than
                     *   1024 blocks each waiting for its NVLink acknowledgements. */
} pcl_handoff;
int pcl_crop_handoff(pcl_handle* h, const pcl_crop_spec* crop, const uint8_t* d_board,
                     int32_t* d_crop_state, const pcl_outputs* out, const pcl_handoff* x,
                     void* stream);

/* Copy the per-env latched error words (PCL_ENV_ERR_*) to d_out i32 [B]. */
int pcl_error_codes(pcl_handle* h, int32_t* d_out, void* stream);

/* Number of kernels this handle has launched so far. */
int pcl_launch_count(pcl_handle* h, int64_t* out);

const char* pcl_status_string(int status);
/* Text of the last CUDA failure behind a PCL_ERR_CUDA of this handle ("" if none);
 * valid until the next failing call on the handle. */
const char* pcl_last_error(pcl_handle* h);
int pcl_abi_version(void);
/* sizeof of the four structs that cross the boundary, for bindings to verify their
 * own layouts at load time: out[0..3] = pcl_spec, pcl_state, pcl_outputs, pcl_crop_spec. */
int pcl_struct_sizes(int32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif  /* PCL_H_ */
