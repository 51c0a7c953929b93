// scrolly_maze.cu — fused step kernel for examples/scrolly_maze.py.
//
// One launch = Engine.play() for every env (engine.py:583-639): the three
// update groups [['#'], ['a','b','c','P'], ['@']] (scrolly_maze.py:241), the
// Plot consultation, and the final z-ordered render 'abc@#P' (:242).
//
// The two intermediate renders of the reference (one per update group,
// engine.py:735) are never materialised: the only board cells the entities
// read between groups are the <= 9 neighbours of a MazeWalker, tested against
// impassable = '#', and in z-order 'abc@#P' a cell shows '#' iff the wall
// curtain covers it and the (previously rendered) player is not standing on
// it.
//
// Memory schedule (one warp per env, everything staged through shared memory):
//   1. records (sprites/drapes/plot, 64 words) -> smem with two coalesced loads (for
//      the write-back); the fields this game uses go straight to registers with
//      16-byte loads issued beside them, not through a store to smem and a read back;
//   2. group 0 ('#' MazeDrape) is pure register arithmetic and fixes BOTH
//      final window corners (the '@' drape can only obey an order, never issue
//      one: by the time it runs, the player's permit is already for frame+1);
//   3. one batch of loads is issued for everything else the step will read:
//        - cp.async: the backdrop tile (issued before anything else) and the
//          two windows of the bit-packed patterns (4 words per row, two 8-byte
//          copies) -> smem, no registers held;
//        - plain loads: a 5x5 patch of wall bits around each of the 4 walkers
//          (covers every cell any _check_motion of this step can consult,
//          wherever the scroll order moves the walker first) and the 3x3 patch
//          of coin bits around the player, one cell per lane, 4 per lane;
//   4. groups 1 and 2 run on registers + ballots of those bits;
//   5. each lane shifts whole window rows once into one word per 16-cell board
//      segment (wall16 << 16 | coin16); the paint loop then composes 16-byte
//      segments from smem (prmt with a 256-entry selector table) and streams them
//      out with uint4 stores; records go back with two coalesced stores.
// So a step costs ~two dependent DRAM round trips (records, then everything).
// The 64 x 64 board has its own instantiation of the same body with the shape fixed
// at compile time (fully unrolled staging / segment / paint loops, constant smem
// offsets); every other shape runs the instantiation that reads it at run time.
//
// Tried and rejected (round 2, A/B on one B200, profiles/r02_step_variants.txt): HALF a
// warp per env (two envs per warp, every warp primitive on the half's 16-lane mask; the
// ~760 warp instructions of game logic per env issued once per two envs).  Bit-exact on
// the whole GPU suite, but 14.2 us per 4096-env step against 11.96 us for this kernel:
// the step is bound by the length of ONE warp's dependent chain, not by issue slots, and
// halving the lanes doubles every staging / paint loop on that chain while 14 instead of
// 28 warps per SM hide less of it.
//
// Sprite order P,a,b,c (indices 0..3); drape order '#','@' (0, 1).
// Registers: patroller aux0 = moving_east; P aux0/aux1 = scroll permit mask /
// permit frame; '@' aux0/aux1 = board cell of a coin already removed from the
// pattern but still on the (not yet refreshed) curtain, or -1; plot aux0 =
// coins left in the pattern.
#include "pcl_device.cuh"
#include "pcl_kernels.cuh"
#include "pcl_crop.cuh"

namespace pcl {

namespace {

constexpr int kS = 4;
constexpr int kWarpsPerBlock = 4;
constexpr int kRecWords = 64;     // 4 sprites * 8 + 2 drapes * 8 + plot 16

__device__ __forceinline__ int action_to_motion(int a) {   // scrolly_maze.py:262-271
  // actions 0..4 = N S W E stay (motion codes 0 4 6 2 8), anything else = no motion:
  // one nibble per action in a constant instead of a chain of selects
  constexpr unsigned kTable = (PCL_M_N) | (PCL_M_S << 4) | (PCL_M_W << 8) | (PCL_M_E << 12) |
                              (PCL_M_STAY << 16);
  return (unsigned)a < 5u ? (int)((kTable >> (4 * a)) & 15u) : PCL_M_NONE;
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::
               "r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
}

__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::
               "r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem));
}

// A 64-cell window row starts at bit corner_c of its pattern row; the four words
// from the even word at or below corner_c >> 5 always cover it (<= 31 + 32 + 64
// bits), and pattern rows are 8-byte aligned (pattern_words is even), so a row is
// staged with two 8-byte cp.async into a 16-byte smem slot.

// prmt.b32 without __byte_perm's selector masking (the table holds nibbles 0..5).
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}

// Words staged per window row: a W-cell window row starts at bit corner_c of its
// pattern row; from the even word at or below corner_c >> 5 it spans at most
// 63 + W bits.  4 words (two 8-byte cp.async, one 16-byte slot) up to W = 64, 6 or 8
// beyond (drapes.py:293-376 puts no limit on the board width).
__host__ __device__ __forceinline__ int window_words(int W) { return 2 * ((63 + W + 63) / 64); }

__host__ __device__ __forceinline__ size_t warp_smem_bytes(int H, int pitch, int nw) {
  // records, backdrop tile, two nw-word window rows per board row, one word per segment
  const size_t rows = (((size_t)H * nw * 4) + 15) & ~(size_t)15;
  return kRecWords * 4 + (size_t)H * pitch + 2 * rows +
         (((size_t)H * (pitch >> 2) + 15) & ~(size_t)15);      // keep every warp's slice 16-byte aligned
}

// Programmatic dependent launch: let the next kernel of the stream begin its
// launch/prologue while this one runs, and wait for everything earlier in the
// stream before touching global memory.
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_wait_prior_grids() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// Selector table of the paint loop (see the kernel): 256 x u16, built at compile
// time and pulled into shared memory with one cp.async per lane of warp 0.
struct SelTable { uint16_t v[256]; };
constexpr SelTable make_sel_table() {
  SelTable t = {};
  for (int idx = 0; idx < 256; ++idx) {
    unsigned sel = 0;
    for (int k = 0; k < 4; ++k) {
      const unsigned nib = ((idx >> (4 + k)) & 1) ? 5u : ((idx >> k) & 1) ? 4u : (unsigned)k;
      sel |= nib << (4 * k);
    }
    t.v[idx] = (uint16_t)sel;
  }
  return t;
}
__device__ __align__(16) const SelTable g_sel = make_sel_table();

// 3x3 "blocked" mask (bit (dr+1)*3 + dc+1, sprites.py:495-507) around the virtual
// position (vrow, vcol) of a walker whose 5x5 wall patch `field` is centred on
// (r0, c0): a cell blocks iff it is on the board, the wall curtain covers it and the
// player is not painted over it (z-order ... '#' 'P').  Pure per-lane arithmetic.
__device__ __forceinline__ unsigned blocked3x3(int vrow, int vcol, int r0, int c0, unsigned field,
                                               int H, int W, bool p_vis, int p_row, int p_col) {
  const int br = vrow - r0 + 1, bc = vcol - c0 + 1;    // 3x3 origin inside the 5x5: 0..2
  if ((unsigned)br > 2u || (unsigned)bc > 2u) return 0u;   // cannot happen (|order|, |move| <= 1)
  unsigned colmask = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) colmask |= ((unsigned)(vcol - 1 + i) < (unsigned)W ? 1u : 0u) << i;
  unsigned blk = 0;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    unsigned bits = (field >> ((br + j) * 5 + bc)) & colmask;
    if ((unsigned)(vrow - 1 + j) >= (unsigned)H) bits = 0;
    blk |= bits << (3 * j);
  }
  const int dr = p_row - vrow + 1, dc = p_col - vcol + 1;
  if (p_vis && (unsigned)dr <= 2u && (unsigned)dc <= 2u) blk &= ~(1u << (dr * 3 + dc));
  return blk;
}

// All eight motions of sprites.py:479-546 at once: bit m set = motion code m is
// legal (N NE E SE S SW W NW), plus STAY.
__device__ __forceinline__ int legal_motions(unsigned b) {
  const unsigned nw = b & 1u, n = (b >> 1) & 1u, ne = (b >> 2) & 1u, w = (b >> 3) & 1u,
                 e = (b >> 5) & 1u, sw = (b >> 6) & 1u, s = (b >> 7) & 1u, se = (b >> 8) & 1u;
  const unsigned blocked = n | ((ne | (n & e)) << 1) | (e << 2) | ((se | (s & e)) << 3) |
                           (s << 4) | ((sw | (s & w)) << 5) | (w << 6) | ((nw | (n & w)) << 7);
  return (int)((~blocked & 0xffu) | (1u << PCL_M_STAY));
}

// drapes.py:487-659 `_maybe_move` when the player is the only possible egocentric
// participant (validated in pcl_create): same decisions as pcl::scrolly_move.
__device__ __forceinline__ void scrolly_move_p(Drape& d, const ScrollyCfg& cfg, int motion,
                                               Plot& plot, int p_row, int p_col, int p_permit,
                                               int p_permit_frame) {
  if (d.last_frame < plot.frame) {
    d.last_frame = plot.frame;
    d.pre_r = d.corner_r; d.pre_c = d.corner_c;
  }
  const int dr = motion_dr(motion), dc = motion_dc(motion);
  if (plot.order_frame == plot.frame) {          // obey an existing order :513-535
    if (dr != plot.order_r && dc != plot.order_c) plot.error |= PCL_ENV_ERR_ORDER_MISMATCH;
    d.corner_r += plot.order_r; d.corner_c += plot.order_c;
    return;
  }
  if (motion == PCL_M_STAY) return;
  const bool ego = plot.ego_mask & 1;
  const bool possible = !ego || (p_permit_frame == plot.frame && ((p_permit >> motion) & 1));
  int orr, occ;
  if (!cfg.have_margins) {                       // :598-623
    if (!possible) return;
    const int nr = d.corner_r + dr, nc = d.corner_c + dc;
    orr = (0 <= nr && nr <= cfg.limit_r) ? dr : 0;
    occ = (0 <= nc && nc <= cfg.limit_c) ? dc : 0;
  } else {                                       // :625-687
    if (!ego) return;
    const int nr = p_row + dr, nc = p_col + dc;  // TRUE position
    const bool want_v = (p_row > nr && nr <= cfg.m_north) || (p_row < nr && nr >= cfg.m_south);
    const bool want_h = (p_col > nc && nc <= cfg.m_west) || (p_col < nc && nc >= cfg.m_east);
    if (!(want_v || want_h)) return;
    orr = want_v ? dr : 0; occ = want_h ? dc : 0;
    const int cr = d.corner_r + orr, cc = d.corner_c + occ;
    if (!((0 <= cr && cr <= cfg.limit_r) && (0 <= cc && cc <= cfg.limit_c)) || !possible) return;
  }
  d.corner_r += orr; d.corner_c += occ;
  plot.order_r = orr; plot.order_c = occ; plot.order_frame = plot.frame;
}

// Phase stamps for tools/step_phases.py: compiled only with -DPCL_STEP_PHASES, nothing
// in the normal build.  Lane 0 of each warp records %globaltimer and clock64() at
// kPhases points of the step (entry, after griddepcontrol.wait, records landed, second
// batch of loads issued, cp.async drained, paint start, paint end) and its %smid.
#ifdef PCL_STEP_PHASES
constexpr int kPhases = 7, kPhaseEnvs = 8192, kPhaseWords = 2 * kPhases + 2;
__device__ unsigned long long g_step_phases[kPhaseEnvs * kPhaseWords];
__device__ __forceinline__ void phase_stamp(int env, int lane, int i) {
  if (lane == 0 && env < kPhaseEnvs) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    unsigned long long* w = g_step_phases + (size_t)env * kPhaseWords;
    w[i] = t;
    w[kPhases + i] = (unsigned long long)clock64();
    if (i == 0) {
      unsigned sm;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
      w[2 * kPhases] = sm;
    }
  }
}
#define PCL_PHASE(i) phase_stamp(env, lane, (i))
#else
#define PCL_PHASE(i) ((void)0)
#endif

// Records: loads of 16 bytes straight from global memory into registers (every lane
// the same address: one request per warp), issued beside the coalesced copy that
// goes to shared memory for the write-back, so no field waits for a store to shared
// memory and a read back.
__device__ __forceinline__ Sprite load_sprite(const int32_t* r) {
  const int4 a = *reinterpret_cast<const int4*>(r), b = *reinterpret_cast<const int4*>(r + 4);
  Sprite s;
  s.row = a.x; s.col = a.y; s.vrow = a.z; s.vcol = a.w;
  s.flags = b.x; s.aux0 = b.y; s.aux1 = b.z; s.aux2 = 0;
  return s;
}
__device__ __forceinline__ Drape load_drape(const int32_t* r) {
  const int4 a = *reinterpret_cast<const int4*>(r), b = *reinterpret_cast<const int4*>(r + 4);
  Drape d;
  d.corner_r = a.x; d.corner_c = a.y; d.pre_r = a.z; d.pre_c = a.w;
  d.last_frame = b.x; d.aux0 = b.y; d.aux1 = b.z; d.aux2 = 0;
  return d;
}
// Plot words 0..8 (frame .. aux0), the ones this game reads.
__device__ __forceinline__ Plot load_plot(const int32_t* r) {
  const int4 a = *reinterpret_cast<const int4*>(r), b = *reinterpret_cast<const int4*>(r + 4);
  Plot pl;
  pl.frame = a.x; pl.game_over = a.y; pl.error = a.z; pl.episodes = a.w;
  pl.order_r = b.x; pl.order_c = b.y; pl.order_frame = b.z; pl.ego_mask = b.w;
  pl.aux0 = r[PCL_P_AUX0];
  return pl;
}

// One body for every board shape.  kH / kW > 0 fix the board at compile time (the
// 64 x 64 board of the generated levels, pitch 64): loop trip counts, shared-memory
// offsets and the window width are then constants and the general-width code is
// gone.  kH = kW = 0 takes the shape from the launch parameters (any other board).
template <int kH, int kW>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, 7)
scrolly_maze_step(const StepParams p) {
  static_assert((kH > 0) == (kW > 0) && kW <= 64 && (kW & 15) == 0, "fixed shape: pitch = W <= 64");
  extern __shared__ __align__(16) uint8_t smem_raw[];
  // Byte-permute selectors for 4 cells at once: index = wall nibble << 4 | coin
  // nibble; selector nibble k picks byte 5 ('#') if wall_k, else byte 4 ('@') if
  // coin_k, else byte k of the backdrop word (z-order ... '@' '#' ...).
  // One copy per WARP: a warp then needs no block barrier before it paints (warps of a
  // block leave at different points: ragged tail, frozen envs).
  __shared__ __align__(16) uint16_t s_sel_all[kWarpsPerBlock][256];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  uint16_t* s_sel = s_sel_all[warp];
  cp_async16(reinterpret_cast<uint8_t*>(s_sel) + lane * 16,
             reinterpret_cast<const uint8_t*>(g_sel.v) + lane * 16);
  pdl_launch_dependents();
  const int env = blockIdx.x * kWarpsPerBlock + warp;
  PCL_PHASE(0);
  const bool live = env < p.B;
  const int H = kH ? kH : p.H, W = kW ? kW : p.W, PWW = p.PWW;
  const int pitch = kW ? kW : p.pitch;
  const int nw = window_words(W);            // staged words per window row (4 for W <= 64)

  uint8_t* my = smem_raw + warp * warp_smem_bytes(H, pitch, nw);
  int32_t* rec = reinterpret_cast<int32_t*>(my);
  uint8_t* s_bd = my + kRecWords * 4;
  uint32_t* s_wall = reinterpret_cast<uint32_t*>(s_bd + (size_t)H * pitch);
  uint32_t* s_coin = s_wall + ((H * nw + 3) & ~3);
  // Everything above ran without touching state earlier kernels may have
  // produced (g_sel is a constant); from here on the kernel reads such state.
  pdl_wait_prior_grids();
  PCL_PHASE(1);
  // An attached cropper reads its corner state at the very end: start that line's trip
  // from DRAM now (a hint, no register held).
  if (p.has_cropper && p.cropper.state && live && lane == 0)
    asm volatile("prefetch.global.L2 [%0];" :: "l"(p.cropper.state + (int64_t)env * 4));
  if (!live) {                 // ragged last block: only the selector copy to drain
    cp_async_wait_all();
    return;
  }
  const int64_t lvl = p.st.d_level ? p.st.d_level[env] : env;   // index of static level data

  int32_t* g_sprites = p.st.d_sprites + (int64_t)env * kS * PCL_SPRITE_WORDS;
  int32_t* g_drapes = p.st.d_drapes + (int64_t)env * 2 * PCL_DRAPE_WORDS;
  int32_t* g_plot = p.st.d_plot + (int64_t)env * PCL_PLOT_WORDS;
  const uint32_t* wall_pat = p.st.d_pattern[0] + lvl * p.st.pattern_bstride[0];
  uint32_t* coin_pat = p.st.d_pattern[1] + (int64_t)env * p.st.pattern_bstride[1];

  // The env's action word does not depend on the records either: issue its load now,
  // beside theirs, instead of one memory round trip later (it is only USED if the env
  // neither restarts nor is frozen).
  int action_early = PCL_ACTION_NONE;
  if (p.mode == MODE_STEP) action_early = p.actions[(int64_t)env * p.actions_per_env];
  // ---- 0. the backdrop tile depends on nothing: get it moving first --------
  {
    const uint8_t* src = p.st.d_backdrop + lvl * p.st.backdrop_bstride + lane * 16;
    uint8_t* dst = s_bd + lane * 16;
    const int n16 = (H * pitch) >> 4;
#pragma unroll(kH ? kH * kW / 512 : 4)
    for (int i = lane; i < n16; i += 32, src += 512, dst += 512) cp_async16(dst, src);
  }
  // ---- 1. records -> registers (the fields this game reads, one lane's walker and
  // the player, drapes and plot in every lane) and -> smem (coalesced, for the
  // write-back and the cropper epilogue) ---------------------------------------
  const int me = lane & 3;                   // ONE walker per lane (P, a, b, c) in group 1
  Sprite mine = load_sprite(g_sprites + me * PCL_SPRITE_WORDS);
  Sprite p0 = load_sprite(g_sprites);        // the player: previous render + permits
  Drape walls = load_drape(g_drapes), coins = load_drape(g_drapes + PCL_DRAPE_WORDS);
  Plot plot = load_plot(g_plot);
  rec[lane] = g_sprites[lane];
  rec[32 + lane] = lane < 16 ? g_drapes[lane] : g_plot[lane - 16];
  bool restart;                              // engine.py:520-581, 619-624
  bool frozen = false;
  if (p.mode == MODE_RESET) {
    restart = (p.env_mask == nullptr) || (p.env_mask[env] != 0);
    frozen = !restart;
  } else {
    restart = plot.game_over && p.auto_reset;
    frozen = plot.game_over && !p.auto_reset;   // reference raises; env stays frozen
  }
  if (frozen) {                              // warp-uniform
    cp_async_wait_all();
    return;
  }
  PCL_PHASE(2);
  int action;
  if (restart) {
    const int episodes = plot.episodes, error = plot.error;
    __syncwarp();
    const int32_t* si = p.st.d_sprites_init + lvl * p.st.sprites_init_bstride;
    const int32_t* di = p.st.d_drapes_init + lvl * p.st.drapes_init_bstride;
    const int32_t* pi = p.st.d_plot_init + lvl * p.st.plot_init_bstride;
    rec[lane] = __ldg(si + lane);
    rec[32 + lane] = lane < 16 ? __ldg(di + lane) : __ldg(pi + lane - 16);
    mine = load_sprite(si + me * PCL_SPRITE_WORDS);
    p0 = load_sprite(si);
    walls = load_drape(di); coins = load_drape(di + PCL_DRAPE_WORDS);
    plot = load_plot(pi);
    plot.error = error;
    // Fresh coins: restore the mutable pattern (one Engine per episode).
    const uint32_t* src = p.st.d_pattern_init[1] + lvl * p.st.pattern_init_bstride[1];
    const int n = p.PH * PWW;
    for (int i = lane; i < n; i += 32) coin_pat[i] = __ldg(src + i);
    __syncwarp();
    if (lane == 0) { rec[48 + PCL_P_EPISODES] = episodes + 1; rec[48 + PCL_P_ERROR] = error; }
    action = PCL_ACTION_NONE;
  } else {
    action = action_early;
  }
  const int p_row = p0.row, p_col = p0.col, p_vrow = p0.vrow, p_vcol = p0.vcol;
  const bool p_vis = visible(p0);
  const int p_permit = p0.aux0, p_permit_frame = p0.aux1;

  const ScrollyCfg wcfg = scrolly_cfg(H, W, p.PH, p.PW, p.margin[0][0], p.margin[0][1]);
  const ScrollyCfg ccfg = scrolly_cfg(H, W, p.PH, p.PW, p.margin[1][0], p.margin[1][1]);
  Directives dir = fresh_directives();
  const int motion = action_to_motion(action);

  plot.frame += 1;                                           // engine.py:716

  // ---- 2. update group 0: '#' MazeDrape (scrolly_maze.py:308-329) --------
  if (motion != PCL_M_NONE)
    scrolly_move_p(walls, wcfg, motion, plot, p_row, p_col, p_permit, p_permit_frame);
  const bool ordered = plot.order_frame == plot.frame;
  const int wr = walls.corner_r, wc = walls.corner_c;
  // Where the '@' window will be after it obeys the same order (checked below).
  const int cr_pred = coins.corner_r + (ordered && motion != PCL_M_NONE ? plot.order_r : 0);
  const int cc_pred = coins.corner_c + (ordered && motion != PCL_M_NONE ? plot.order_c : 0);

  // ---- 3. one batch of loads ---------------------------------------------
  const int we = (wc >> 5) & ~1, ce = (cc_pred >> 5) & ~1;   // first staged word (even)
  const bool narrow = W <= 64;               // the 4-word fast paths (pitch <= 64)
  if (narrow) {
    const int nhalf = H * 2;                 // two 8-byte halves per window row
#pragma unroll
    for (int i = lane; i < nhalf; i += 32) {
      const int r = i >> 1, k = (i & 1) * 2;
      cp_async8(s_wall + i * 2, wall_pat + (int64_t)(wr + r) * PWW + we + k);
      cp_async8(s_coin + i * 2, coin_pat + (int64_t)(cr_pred + r) * PWW + ce + k);
    }
  } else {                                   // boards wider than 64 columns
    const int hw = nw >> 1, nhalf = H * hw;
    for (int i = lane; i < nhalf; i += 32) {
      const int r = i / hw, k = (i - r * hw) * 2;
      cp_async8(s_wall + i * 2, wall_pat + (int64_t)(wr + r) * PWW + we + k);
      cp_async8(s_coin + i * 2, coin_pat + (int64_t)(cr_pred + r) * PWW + ce + k);
    }
  }
  PCL_PHASE(3);
  scrolly_touch_prescroll(coins, plot);      // '@' has not moved yet this frame
  // Look-up bits, one pattern ROW per lane: lanes 0..19 = row k of the 5x5 wall
  // patch of walker w (lane = 5 w + k; covers every cell any _check_motion of this
  // step can consult, wherever the scroll order moves the walker first), lanes
  // 20..22 = the 3 rows of the coin patch around the player, lane 23 = the coin
  // bit at the pre-scroll corner (an off-board player sits at (0, 0)).
  unsigned rowbits = 0;
  {
    const uint32_t* row = nullptr;
    int c_first = 0, limit = 0;              // first pattern column, words in the row
    const int w = min(lane / 5, 3), k = lane - w * 5;      // lane w holds walker w
    const int w_vrow = __shfl_sync(PCL_FULL, mine.vrow, w), w_vcol = __shfl_sync(PCL_FULL, mine.vcol, w);
    if (lane < 20) {
      const int pr = wr + w_vrow + k - 2;
      c_first = wc + w_vcol - 2;
      if ((unsigned)pr < (unsigned)p.PH) { row = wall_pat + (int64_t)pr * PWW; limit = PWW; }
    } else if (lane < 23) {
      const int r = p_vrow + (lane - 20) - 1;
      c_first = coins.pre_c + p_vcol - 1;
      if ((unsigned)r < (unsigned)H) { row = coin_pat + (int64_t)(coins.pre_r + r) * PWW; limit = PWW; }
    } else if (lane == 23) {
      c_first = coins.pre_c;
      row = coin_pat + (int64_t)coins.pre_r * PWW; limit = PWW;
    }
    if (row != nullptr) {
      const int wi = c_first >> 5;           // floor, may be -1
      const uint32_t lo = (unsigned)wi < (unsigned)limit ? row[wi] : 0u;
      const uint32_t hi = (unsigned)(wi + 1) < (unsigned)limit ? row[wi + 1] : 0u;
      rowbits = __funnelshift_r(lo, hi, c_first & 31) & 31u;
    }
  }
  // Pattern columns past PW are zero padding and negative ones read as zero, so
  // the wall bits need no further masking; coin bits are masked to the board.
  unsigned field = 0;                        // my walker's 5x5 patch, bit (dr+2)*5 + dc+2
#pragma unroll
  for (int k = 0; k < 5; ++k) field |= __shfl_sync(PCL_FULL, rowbits, me * 5 + k) << (5 * k);
  unsigned coin9 = 0;                        // 3x3 around the player's start + the (0,0) cell
  {
    unsigned colmask = 0;
#pragma unroll
    for (int i = 0; i < 3; ++i)
      colmask |= ((unsigned)(p_vcol - 1 + i) < (unsigned)W ? 1u : 0u) << i;
#pragma unroll
    for (int k = 0; k < 3; ++k) coin9 |= (__shfl_sync(PCL_FULL, rowbits, 20 + k) & colmask) << (3 * k);
    coin9 |= (__shfl_sync(PCL_FULL, rowbits, 23) & 1u) << 9;
  }

  // ---- 4a. update group 1: patrollers a, b, c then P, ONE WALKER PER LANE ----
  // The four walkers do not interact within a frame: each reads the board of
  // render #1 (walls at the new corner, P painted where the previous render put it)
  // and the shared plot; P moves last, so patrollers compare with its OLD virtual
  // position.  (sprites.py:356-477, scrolly_maze.py:258-305.)
  const int r0 = mine.vrow, c0 = mine.vcol;
  const bool is_p = me == 0;
  const bool even = (plot.frame % 2) == 0;
  if (even) scrolly_touch_prescroll(walls, plot);           // PatrollerSprite :291
  int my_err = 0;
  bool hit = false;
  int mot;                                   // this lane's motion this frame
  if (is_p) {
    mot = motion;                            // PCL_M_NONE: P does not move at all (:258)
  } else if (!even) {
    mot = PCL_M_STAY;
  } else {
    const int step = mine.aux0 ? 1 : -1;
    int pr = r0 + walls.pre_r, pc = c0 + walls.pre_c + step;
    bool next_to_wall = false;
    if ((unsigned)pr < (unsigned)p.PH && (unsigned)pc < (unsigned)p.PW) {
      // Same cell seen from the post-scroll corner: inside the 5x5 patch.
      const int dr = pr - wr - r0 + 2, dc = pc - wc - c0 + 2;
      next_to_wall = (field >> (dr * 5 + dc)) & 1u;
    } else {
      // NumPy indexing: negatives wrap once, anything else is an IndexError.
      if (pr < 0) pr += p.PH;
      if (pc < 0) pc += p.PW;
      if ((unsigned)pr < (unsigned)p.PH && (unsigned)pc < (unsigned)p.PW)
        next_to_wall = bit_at(wall_pat + (int64_t)pr * PWW, pc);
      else
        my_err |= PCL_ENV_ERR_INDEX;
    }
    if (next_to_wall) mine.aux0 = !mine.aux0;
    mot = mine.aux0 ? PCL_M_E : PCL_M_W;
  }
  if (mot != PCL_M_NONE) {                   // sprites.py:356-389 `_move`
    const int dr = motion_dr(mot), dc = motion_dc(mot);
    if (ordered) {                           // _obey_scrolling_order :413-454
      walker_teleport(mine, H, W, mine.vrow - plot.order_r, mine.vcol - plot.order_c);
      if (is_p && plot.order_r != dr && plot.order_c != dc) my_err |= PCL_ENV_ERR_ORDER_MISMATCH;
    }
    bool legal = true;
    unsigned blk = 0;
    if (mot != PCL_M_STAY || is_p) {
      blk = blocked3x3(mine.vrow, mine.vcol, r0, c0, field, H, W, p_vis, p_row, p_col);
      legal = motion_legal(blk, mot);
    }
    if (legal && mot != PCL_M_STAY) {
      walker_teleport(mine, H, W, mine.vrow + dr, mine.vcol + dc);      // _raw_move :391
      if (is_p) blk = blocked3x3(mine.vrow, mine.vcol, r0, c0, field, H, W, p_vis, p_row, p_col);
    }
    if (is_p) {                              // :456-477 + scrolling.py:373-434
      const int valid_at = plot.frame + 1;
      if (mine.aux1 != valid_at) { mine.aux1 = valid_at; mine.aux0 = 0; }
      mine.aux0 |= legal_motions(blk);
    } else if (even) {
      hit = mine.vrow == p_vrow && mine.vcol == p_vcol;     // PatrollerSprite :303-305
    }
  }
  __syncwarp();                              // every lane has read the records it needs (racecheck)
  if (lane < 4) {                            // write my walker back
    int32_t* r = rec + me * PCL_SPRITE_WORDS;
    r[PCL_S_ROW] = mine.row; r[PCL_S_COL] = mine.col;
    r[PCL_S_VROW] = mine.vrow; r[PCL_S_VCOL] = mine.vcol;
    r[PCL_S_FLAGS] = mine.flags; r[PCL_S_AUX0] = mine.aux0;
    if (is_p) r[PCL_S_AUX1] = mine.aux1;
  }
  if (motion != PCL_M_NONE) plot.ego_mask |= 1;             // sprites.py:443 (P only)
  plot.error |= __reduce_or_sync(PCL_FULL, (unsigned)(lane < 4 ? my_err : 0));
  if (__any_sync(PCL_FULL, lane < 4 && hit)) terminate(dir);
  // The player after its move, for everything below.
  Sprite pl;
  pl.row = __shfl_sync(PCL_FULL, mine.row, 0); pl.col = __shfl_sync(PCL_FULL, mine.col, 0);
  pl.vrow = __shfl_sync(PCL_FULL, mine.vrow, 0); pl.vcol = __shfl_sync(PCL_FULL, mine.vcol, 0);
  pl.flags = __shfl_sync(PCL_FULL, mine.flags, 0);
  pl.aux0 = __shfl_sync(PCL_FULL, mine.aux0, 0); pl.aux1 = __shfl_sync(PCL_FULL, mine.aux1, 0);

  // ---- 4b. update group 2: '@' CashDrape (scrolly_maze.py:341-364) -------
  int picked_r = -1, picked_c = -1;          // pattern cell cleared this frame
  {
    const int dr = pl.row - p_vrow, dc = pl.col - p_vcol;
    bool coin;
    const int pr = coins.pre_r + pl.row, pc = coins.pre_c + pl.col;
    if (pl.row == 0 && pl.col == 0 && !on_board(pl.vrow, pl.vcol, H, W))
      coin = (coin9 >> 9) & 1u;              // off-board player sits at (0, 0)
    else if ((unsigned)(dr + 1) <= 2u && (unsigned)(dc + 1) <= 2u)
      coin = (coin9 >> ((dr + 1) * 3 + dc + 1)) & 1u;
    else
      coin = bit_at(coin_pat + (int64_t)pr * PWW, pc);   // cannot happen
    if (coin) {
      add_reward(dir, 100);
      if (lane == 0) coin_pat[(int64_t)pr * PWW + (pc >> 5)] &= ~(1u << (pc & 31));
      picked_r = pr; picked_c = pc;
      plot.aux0 -= 1;
      if (plot.aux0 == 0) terminate(dir);
      coins.aux0 = pl.row; coins.aux1 = pl.col;         // stale until next refresh
    }
  }
  if (motion != PCL_M_NONE) {
    scrolly_move_p(coins, ccfg, motion, plot, pl.row, pl.col, pl.aux0, pl.aux1);
    coins.aux0 = -1; coins.aux1 = -1;                    // _update_curtain :689
  } else if (action == 5) {
    terminate(dir);
  }

  // ---- _apply_and_clear_plot (engine.py:761-847); no z-order changes here.
  cp_async_wait_all();
  PCL_PHASE(4);
  __syncwarp();
  if (lane == 0) {
    int32_t* r = rec + 32;
    r[PCL_D_CORNER_R] = walls.corner_r; r[PCL_D_CORNER_C] = walls.corner_c;
    r[PCL_D_PRE_R] = walls.pre_r; r[PCL_D_PRE_C] = walls.pre_c;
    r[PCL_D_LAST_FRAME] = walls.last_frame;
    r += PCL_DRAPE_WORDS;
    r[PCL_D_CORNER_R] = coins.corner_r; r[PCL_D_CORNER_C] = coins.corner_c;
    r[PCL_D_PRE_R] = coins.pre_r; r[PCL_D_PRE_C] = coins.pre_c;
    r[PCL_D_LAST_FRAME] = coins.last_frame;
    r[PCL_D_AUX0] = coins.aux0; r[PCL_D_AUX1] = coins.aux1;
    r = rec + 48;
    r[PCL_P_FRAME] = plot.frame; r[PCL_P_GAME_OVER] = dir.game_over;
    r[PCL_P_ERROR] = plot.error;
    r[PCL_P_ORDER_R] = plot.order_r; r[PCL_P_ORDER_C] = plot.order_c;
    r[PCL_P_ORDER_FRAME] = plot.order_frame; r[PCL_P_EGO_MASK] = plot.ego_mask;
    r[PCL_P_AUX0] = plot.aux0;
    p.out.d_reward[env] = dir.reward;
    p.out.d_has_reward[env] = (uint8_t)dir.has_reward;
    p.out.d_discount[env] = dir.discount;
    p.out.d_done[env] = (uint8_t)dir.game_over;
    // The coin window was staged before the pick-up: clear the bit there too.
    if (picked_r >= 0) {
      const int r2 = picked_r - cr_pred, b = picked_c - (ce << 5);
      if ((unsigned)r2 < (unsigned)H && (unsigned)b < (unsigned)(nw * 32))
        s_coin[r2 * nw + (b >> 5)] &= ~(1u << (b & 31));
    }
  }
  const int cr = coins.corner_r, cc = coins.corner_c;
  int ce_final = ce;
  if (cr != cr_pred || cc != cc_pred) {      // '@' issued its own order: restage
    __syncwarp();
    ce_final = (cc >> 5) & ~1;
    for (int i = lane; i < H * nw; i += 32)
      s_coin[i] = coin_pat[(int64_t)(cr + i / nw) * PWW + ce_final + i % nw];
  }
  __syncwarp();
  g_sprites[lane] = rec[lane];
  if (lane < 16) g_drapes[lane] = rec[32 + lane];
  else g_plot[lane - 16] = rec[32 + lane];

  // ---- 5. final render, z-order a b c @ # P (engine.py:737-759) ----------
  // 5a. Window rows -> ONE word per 16-cell board segment (wall16 << 16 | coin16),
  // aligned to the board: each lane shifts whole rows once, so the streaming loop
  // below does no bit addressing at all.  Cells past W and the stale coin
  // (drapes.py:689 has not refreshed the curtain yet) are folded in here.
  const int spr = pitch >> 4;                // 16-byte segments per row
  uint32_t* s_seg = s_coin + ((H * nw + 3) & ~3);
  const int wsh = wc - (we << 5), csh = cc - (ce_final << 5);     // 0..63 into the staged row
  if (narrow) {
    const uint32_t m_lo = W >= 32 ? 0xffffffffu : (1u << W) - 1u;
    const uint32_t m_hi = W >= 64 ? 0xffffffffu : W > 32 ? (1u << (W - 32)) - 1u : 0u;
#pragma unroll
    for (int r = lane; r < H; r += 32) {
      const uint4 wv = *reinterpret_cast<const uint4*>(s_wall + r * 4);
      const uint4 cv = *reinterpret_cast<const uint4*>(s_coin + r * 4);
      const uint32_t wa = (wsh & 32) ? wv.y : wv.x, wb = (wsh & 32) ? wv.z : wv.y,
                     wd = (wsh & 32) ? wv.w : wv.z;
      const uint32_t ca = (csh & 32) ? cv.y : cv.x, cb = (csh & 32) ? cv.z : cv.y,
                     cd = (csh & 32) ? cv.w : cv.z;
      const uint32_t w_lo = __funnelshift_r(wa, wb, wsh & 31) & m_lo;
      const uint32_t w_hi = __funnelshift_r(wb, wd, wsh & 31) & m_hi;
      const uint32_t c_lo = __funnelshift_r(ca, cb, csh & 31) & m_lo;
      const uint32_t c_hi = __funnelshift_r(cb, cd, csh & 31) & m_hi;
      uint32_t* out = s_seg + r * spr;
      out[0] = __byte_perm(c_lo, w_lo, 0x5410);
      if (spr > 1) out[1] = __byte_perm(c_lo, w_lo, 0x7632);
      if (spr > 2) out[2] = __byte_perm(c_hi, w_hi, 0x5410);
      if (spr > 3) out[3] = __byte_perm(c_hi, w_hi, 0x7632);
    }
  } else {                                   // general width: one (row, segment) per lane and round
    for (int i = lane; i < H * spr; i += 32) {
      const int r = i / spr, j = i - r * spr;
      const int ncols = min(16, W - 16 * j);
      if (ncols <= 0) { s_seg[i] = 0; continue; }          // pitch padding past the board
      const uint32_t keep = (1u << ncols) - 1u;
      const int wo = wsh + 16 * j, co = csh + 16 * j;
      const uint32_t* wrow = s_wall + r * nw;
      const uint32_t* crow = s_coin + r * nw;
      // the second word is only fetched while inside the staged row
      const uint32_t w16 = __funnelshift_r(wrow[wo >> 5], (wo >> 5) + 1 < nw ? wrow[(wo >> 5) + 1] : 0u,
                                           wo & 31) & keep;
      const uint32_t c16 = __funnelshift_r(crow[co >> 5], (co >> 5) + 1 < nw ? crow[(co >> 5) + 1] : 0u,
                                           co & 31) & keep;
      s_seg[i] = (w16 << 16) | c16;
    }
  }
  // a, b, c lie under both drapes, so they are patched into the staged backdrop
  // up front, in z-order (a lane each, one after the other); the player is the TOP
  // layer: its character also goes into the staged tile, and both drape bits of its
  // cell are cleared so that the compose below keeps the tile's byte there — the
  // streaming loop then has no sprite test at all.
  __syncwarp();
  if (lane == 0 && coins.aux0 >= 0)
    s_seg[coins.aux0 * spr + (coins.aux1 >> 4)] |= 1u << (coins.aux1 & 15);
#pragma unroll
  for (int i = 1; i < kS; ++i) {
    if (lane == i && visible(mine)) s_bd[mine.row * pitch + mine.col] = p.sprite_char[i];
    __syncwarp();
  }
  if (lane == 0 && visible(pl)) {
    s_bd[pl.row * pitch + pl.col] = p.sprite_char[0];
    s_seg[pl.row * spr + (pl.col >> 4)] &= ~(0x00010001u << (pl.col & 15));
  }
  __syncwarp();                              // (also: this warp's s_sel copy has landed, waited above)
  // 5b. The streaming loop: 16 cells per lane per iteration, segment index ==
  // 16-byte index into both the staged tile and the board (pitch = 16 * spr).
  PCL_PHASE(5);
  const int total = H * spr;
  const unsigned drape_chars = ('#' << 8) | '@';           // bytes 4 and 5 of the permute
  const uint4* src = reinterpret_cast<const uint4*>(s_bd);
  uint4* dst = reinterpret_cast<uint4*>(p.out.d_board + (int64_t)env * H * pitch);
#pragma unroll
  for (int seg = lane; seg < total; seg += 32) {
    uint4 px = src[seg];
    const uint32_t bits = s_seg[seg];
    px.x = prmt(px.x, drape_chars, s_sel[((bits >> 12) & 0xf0u) | (bits & 0xfu)]);
    px.y = prmt(px.y, drape_chars, s_sel[((bits >> 16) & 0xf0u) | ((bits >> 4) & 0xfu)]);
    px.z = prmt(px.z, drape_chars, s_sel[((bits >> 20) & 0xf0u) | ((bits >> 8) & 0xfu)]);
    px.w = prmt(px.w, drape_chars, s_sel[((bits >> 24) & 0xf0u) | ((bits >> 12) & 0xfu)]);
    dst[seg] = px;
  }
  PCL_PHASE(6);
  // ---- 6. an attached cropper (pcl_attach_cropper): the egocentric view of the board
  // this warp has just stored, without a second kernel (ScrollingCropper.crop,
  // cropping.py:393-426).
  if (p.has_cropper) {
    __syncwarp();
    crop_epilogue(p.cropper, p.out.d_board, env, lane, rec, rec + 48);
  }
}

}  // namespace

#ifdef PCL_STEP_PHASES
// Copies the stamps of the last launch: kPhaseEnvs rows of kPhaseWords u64 (globaltimer
// x kPhases, clock64 x kPhases, smid, unused).  Exists only in the stamped build.
extern "C" int pcl_step_phases_read(void* host, size_t bytes) {
  if (bytes > sizeof(g_step_phases)) bytes = sizeof(g_step_phases);
  return (int)cudaMemcpyFromSymbol(host, g_step_phases, bytes);
}
#endif

cudaError_t launch_scrolly_maze(const StepParams& p, cudaStream_t s) {
  if (p.PWW & 1) return cudaErrorInvalidValue;   // window rows are staged in 8-byte halves
  const int blocks = (p.B + kWarpsPerBlock - 1) / kWarpsPerBlock;
  const size_t smem = warp_smem_bytes(p.H, p.pitch, window_words(p.W)) * kWarpsPerBlock;
  if (smem > 227 * 1024) return cudaErrorInvalidValue;         // board too large for one CTA
  // The 64 x 64 board (pitch 64) has its own instantiation; every other shape runs
  // the one that reads the shape from `p`.
  void (*kernel)(const StepParams) = (p.H == 64 && p.W == 64 && p.pitch == 64)
                                         ? scrolly_maze_step<64, 64> : scrolly_maze_step<0, 0>;
  if (smem > 48 * 1024) {   // opt in per launch: the attribute is per device, handles are not
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return e;
  }
  // Programmatic dependent launch: this kernel may start (prologue only) before
  // the previous kernel of the stream has drained; it calls griddepcontrol.wait
  // before its first global access.
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(blocks);
  cfg.blockDim = dim3(kWarpsPerBlock * 32);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, p);
}

}  // namespace pcl
