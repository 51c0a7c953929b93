// box_world.cu — fused step kernel for examples/research/box_world/box_world.py:127-271.
//
// One update group [player] + sorted(drapes), z-order sorted(drapes) + [player]
// (box_world.py:398-400), so every entity reads the board of the previous step's
// final render.  The drapes never overlap and the backdrop is a room of ' ' walled by
// '#', so that board is the backdrop, then the cell plane, then the player:
//
//   plane (pcl_state.d_bits[0], u8 [rows, pitch]): byte = character of the key ('a'..'t'),
//     lock ('A'..'T') or gem ('*') drape covering the cell, 0 = none; bit 7 marks a
//     distractor lock cell (box_world.py:375-376).  Cell (0, 0) is the inventory: the
//     key held, painted over the border '#' (box_world.py:249-251).
//   player: sprite record; AUX0 = move actions taken (_step_counter), AUX1 = max_num_steps.
//
//   PlayerSprite.update (:163-202), actions 0..3 = N S W E only:
//     reward 0; target = the stale board one cell away; '#' refuses the move, ' ' moves,
//     a lock moves only with its key held, a key or the gem only without a lock of any
//     character to its right (BoxThing.is_locked_at, :212-219); after max_num_steps + 1
//     move actions the episode ends.
//   The drape whose character the player stepped onto (where_player_over_me, :221-229):
//     gem  +10 and terminate                                               (:235-238)
//     key  clear the cell, hold the key (dropping the one held)            (:244-251)
//     lock clear the cell, use up the key held; distractor -1 and terminate, else +1 (:261-271)
//   the_plot['over_this'] is never cleared upstream, but a stale entry cannot fire again:
//   its cell was cleared, and curtains only ever gain a cell at (0, 0).
//
// Level rotation (program_arg[1] = stride > 0, program_arg[2] = levels): an AUTO-reset
// moves the env to level (d_level[env] + stride) % levels before it restores the
// templates; pcl_reset restarts the same level.
//
// One warp per env.  Boards up to 32 x 32 (pitch <= 32): at most 64 16-byte row
// segments, two per lane.  The running step loads the records and the live plane in
// one round trip; the three plane bytes the rules read (target, its right neighbour,
// (0, 0)) come from the owning lanes by shuffle.  The backdrop is not loaded: lowering
// admits only the walled room, which the render synthesises.
#include "pcl_device.cuh"
#include "pcl_kernels.cuh"

namespace pcl {

namespace {

constexpr int kWarpsPerBlock = 4;
constexpr int kSlots = 2;                 // 16-byte plane segments per lane

// The plane segments a lane holds, as 4 words each: word i = bytes 4i..4i+3 of slot i / 4.
struct Planes {
  uint32_t w[kSlots * 4];
};

// Byte (r, c) of the plane, from the lane that holds it (warp-uniform r, c).
__device__ __forceinline__ uint32_t plane_byte(const Planes& pl, int r, int c, int spr) {
  const int seg = r * spr + (c >> 4);
  const int idx = ((seg >> 5) << 2) | ((c & 15) >> 2);
  uint32_t v = 0;
#pragma unroll
  for (int i = 0; i < kSlots * 4; ++i) v = (i == idx) ? pl.w[i] : v;
  v = __shfl_sync(PCL_FULL, v, seg & 31);
  return (v >> ((c & 3) * 8)) & 0xffu;
}

// Set byte (r, c) in the holding lane's registers.
__device__ __forceinline__ void plane_set(Planes& pl, int lane, int r, int c, int spr,
                                          uint32_t value) {
  const int seg = r * spr + (c >> 4);
  if ((seg & 31) != lane) return;
  const int idx = ((seg >> 5) << 2) | ((c & 15) >> 2);
  const int sh = (c & 3) * 8;
#pragma unroll
  for (int i = 0; i < kSlots * 4; ++i)
    if (i == idx) pl.w[i] = (pl.w[i] & ~(0xffu << sh)) | (value << sh);
}

__device__ __forceinline__ void load_planes(Planes& pl, const uint8_t* src, int lane, int total) {
#pragma unroll
  for (int k = 0; k < kSlots; ++k) {
    const int s = lane + 32 * k;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (s < total) v = reinterpret_cast<const uint4*>(src)[s];
    pl.w[4 * k] = v.x; pl.w[4 * k + 1] = v.y; pl.w[4 * k + 2] = v.z; pl.w[4 * k + 3] = v.w;
  }
}

__device__ __forceinline__ bool is_lock(uint32_t ch) { return ch - 'A' < 20u; }
__device__ __forceinline__ bool is_key(uint32_t ch) { return ch - 'a' < 20u; }

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
box_world_step(const StepParams p) {
  const int lane = threadIdx.x & 31;
  const int env = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (env >= p.B) return;
  const int H = p.H, W = p.W;
  const int spr = p.pitch >> 4, total = H * spr;
  int32_t* g_sprite = p.st.d_sprites + (int64_t)env * PCL_SPRITE_WORDS;
  int32_t* g_plot = p.st.d_plot + (int64_t)env * PCL_PLOT_WORDS;
  uint8_t* g_plane = reinterpret_cast<uint8_t*>(p.st.d_bits[0] + (int64_t)env * p.st.bits_bstride[0]);

  // ---- loads of a running step, issued together: records and the live plane
  const int4 s0 = reinterpret_cast<const int4*>(g_sprite)[0];
  const int4 s1 = reinterpret_cast<const int4*>(g_sprite)[1];
  const int was_over = g_plot[PCL_P_GAME_OVER];
  int frame = g_plot[PCL_P_FRAME];
  const int error = g_plot[PCL_P_ERROR];
  const int episodes0 = g_plot[PCL_P_EPISODES];
  Planes pl;
  load_planes(pl, g_plane, lane, total);

  bool restart;
  if (p.mode == MODE_RESET) {
    restart = (p.env_mask == nullptr) || (p.env_mask[env] != 0);
    if (!restart) return;
  } else {
    restart = was_over && p.auto_reset;
    if (was_over && !p.auto_reset) return;           // reference raises; env stays frozen
  }
  Sprite pc;
  pc.row = s0.x; pc.col = s0.y; pc.vrow = s0.z; pc.vcol = s0.w;
  pc.flags = s1.x; pc.aux0 = s1.y; pc.aux1 = s1.z; pc.aux2 = 0;
  if (restart) {
    int64_t lvl = env;
    if (p.st.d_level) {
      int l = p.st.d_level[env];
      const int stride = p.program_arg[1];
      if (p.mode == MODE_STEP && stride > 0) {
        l = (int)(((int64_t)l + stride) % p.program_arg[2]);
        __syncwarp();                                 // every lane has read the old index
        if (lane == 0) p.st.d_level[env] = l;
      }
      lvl = l;
    }
    const int32_t* t_s = p.st.d_sprites_init + lvl * p.st.sprites_init_bstride;
    const int32_t* t_p = p.st.d_plot_init + lvl * p.st.plot_init_bstride;
    const int4 t0 = reinterpret_cast<const int4*>(t_s)[0];
    const int4 t1 = reinterpret_cast<const int4*>(t_s)[1];
    frame = t_p[PCL_P_FRAME];
    load_planes(pl, reinterpret_cast<const uint8_t*>(p.st.d_bits_init[0] +
                                                     lvl * p.st.bits_init_bstride[0]),
                lane, total);
    pc.row = t0.x; pc.col = t0.y; pc.vrow = t0.z; pc.vcol = t0.w;
    pc.flags = t1.x; pc.aux0 = t1.y; pc.aux1 = t1.z;
  }
  frame += 1;                                         // engine.py:716
  const int episodes = episodes0 + (restart ? 1 : 0);
  const int action = restart ? PCL_ACTION_NONE : p.actions[(int64_t)env * p.actions_per_env];
  Directives dir = fresh_directives();

  // ---- game logic, warp-uniform
  int changed_r = -1, changed_c = 0;                  // target cell cleared by this step
  uint32_t new_held = 0;
  if ((unsigned)action < 4u) {                        // actions in range(4), :168
    add_reward(dir, 0);                               // REWARD_STEP
    const int dr = action == 0 ? -1 : action == 1 ? 1 : 0;
    const int dc = action == 2 ? -1 : action == 3 ? 1 : 0;
    const int tr = pc.row + dr, tc = pc.col + dc;
    const uint32_t t = plane_byte(pl, tr, tc, spr);
    const uint32_t held = plane_byte(pl, 0, 0, spr);
    const uint32_t right = plane_byte(pl, tr, tc + 1, spr) & 0x7fu;
    const uint32_t tch = t & 0x7fu;
    const bool wall = tr == 0 || tr == H - 1 || tc == 0 || tc == W - 1;
    bool moved;
    if (tch == 0) moved = !wall;                      // ' ' moves, '#' is impassable
    else if (is_lock(tch)) moved = held == tch + ('a' - 'A');
    else moved = !is_lock(right);
    if (moved) { pc.row = pc.vrow = tr; pc.col = pc.vcol = tc; }
    pc.aux0 += 1;
    if (pc.aux0 > pc.aux1) terminate(dir);            // :197-198
    if (moved && tch) {
      if (is_key(tch)) {
        changed_r = tr; changed_c = tc; new_held = tch;
      } else if (is_lock(tch)) {
        changed_r = tr; changed_c = tc; new_held = 0;
        if (t & 0x80u) { add_reward(dir, -1); terminate(dir); }
        else add_reward(dir, 1);
      } else {                                        // the gem
        add_reward(dir, 10);
        terminate(dir);
      }
    }
  }

  // ---- write-back: the whole plane on a restart, else the (at most two) changed bytes
  if (changed_r >= 0) {
    plane_set(pl, lane, changed_r, changed_c, spr, 0u);
    plane_set(pl, lane, 0, 0, spr, new_held);
    if (lane == 0) {
      g_plane[changed_r * p.pitch + changed_c] = 0;
      g_plane[0] = (uint8_t)new_held;
    }
  }
  if (restart) {
#pragma unroll
    for (int k = 0; k < kSlots; ++k) {
      const int s = lane + 32 * k;
      if (s < total)
        reinterpret_cast<uint4*>(g_plane)[s] =
            make_uint4(pl.w[4 * k], pl.w[4 * k + 1], pl.w[4 * k + 2], pl.w[4 * k + 3]);
    }
  }
  if (lane == 0) {
    reinterpret_cast<int4*>(g_sprite)[0] = make_int4(pc.row, pc.col, pc.vrow, pc.vcol);
    reinterpret_cast<int4*>(g_sprite)[1] = make_int4(pc.flags, pc.aux0, pc.aux1, 0);
    g_plot[PCL_P_FRAME] = frame; g_plot[PCL_P_GAME_OVER] = dir.game_over;
    g_plot[PCL_P_EPISODES] = episodes; g_plot[PCL_P_ERROR] = error;
    p.out.d_reward[env] = dir.reward;
    p.out.d_has_reward[env] = (uint8_t)dir.has_reward;
    p.out.d_discount[env] = dir.discount;
    p.out.d_done[env] = (uint8_t)dir.game_over;
  }

  // ---- render (engine.py:737-759): the walled room, the plane, the player
  uint8_t* board = p.out.d_board + (int64_t)env * H * p.pitch;
  const uint32_t player = p.sprite_char[0];
#pragma unroll
  for (int k = 0; k < kSlots; ++k) {
    const int s = lane + 32 * k;
    if (s >= total) continue;
    const int r = s / spr;
    const int c0 = (s - r * spr) << 4;
    const bool edge_row = r == 0 || r == H - 1;
    uint32_t out[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      uint32_t bd = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = c0 + 4 * w + j;
        const uint32_t ch = c >= W ? 0u : (edge_row || c == 0 || c == W - 1) ? '#' : ' ';
        bd |= ch << (8 * j);
      }
      const uint32_t v = pl.w[4 * k + w];
      const uint32_t m = __vcmpne4(v, 0u);            // 0xff where a drape covers the cell
      out[w] = (bd & ~m) | (v & 0x7f7f7f7fu & m);
    }
    const unsigned pm = sprite_bit(pc, r, c0);
    uint4 px = make_uint4(out[0], out[1], out[2], out[3]);
    if (pm) paint_bits(px, pm, player);
    reinterpret_cast<uint4*>(board)[s] = px;
  }
}

}  // namespace

cudaError_t launch_box_world(const StepParams& p, cudaStream_t s) {
  const int blocks = (p.B + kWarpsPerBlock - 1) / kWarpsPerBlock;
  box_world_step<<<blocks, kWarpsPerBlock * 32, 0, s>>>(p);
  return cudaGetLastError();
}

}  // namespace pcl
