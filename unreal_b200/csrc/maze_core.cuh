// Integer core of the maze (host+device so the CPU test harness can exercise it).
// Restates environment/maze_environment.py:66-122 of the reference.
#pragma once
#include "common.cuh"

namespace unreal {

struct MazeLayout {
  uint32_t wall_rows[UNREAL_MAZE_GRID];  // bit x of wall_rows[y] = cell (x,y) is '+'
  int32_t start_x, start_y, goal_x, goal_y;
};

// Host copies of the process-wide map (maze.cu) for kernels of other translation units: the layout K1 steps with
// (evaluate.cu), and its walls as 49 bits, bit cy*7 + cx (the render-fused conv1 kernels of conv_tcgen05.cu).
MazeLayout maze_layout_host();
uint64_t maze_walls49();

struct MazeStep {
  int x1, y1;     // cell after the move (before any reset)
  int reward;     // +1 goal, -1 hit, 0 otherwise
  int terminal;
};

// _move (:76-91) + action decoding (:99-108) + reward/terminal (:114-122)
UNREAL_HD MazeStep maze_step_core(const MazeLayout& L, int x, int y, int action) {
  int dx = (action == 3) - (action == 2);
  int dy = (action == 1) - (action == 0);
  int nx = x + dx, ny = y + dy;
  bool clamped = false;
  if (nx < 0) { nx = 0; clamped = true; } else if (nx > UNREAL_MAZE_GRID - 1) { nx = UNREAL_MAZE_GRID - 1; clamped = true; }
  if (ny < 0) { ny = 0; clamped = true; } else if (ny > UNREAL_MAZE_GRID - 1) { ny = UNREAL_MAZE_GRID - 1; clamped = true; }
  bool hit = clamped;
  if ((L.wall_rows[ny] >> nx) & 1u) { nx = x; ny = y; hit = true; }
  MazeStep s;
  s.x1 = nx; s.y1 = ny;
  s.terminal = (nx == L.goal_x && ny == L.goal_y) ? 1 : 0;
  s.reward = s.terminal ? 1 : (hit ? -1 : 0);
  return s;
}

// Pixels shared by pool block i (cropped rows 4i+2..4i+5) and maze cell c (rows 12c..12c+11):
// 4 for i in {3c, 3c+1}, 2 for i in {3c-1, 3c+2}, else 0   (environment.py:88-99 on two disjoint
// 12x12 squares; SURVEY.md 8a).
UNREAL_HD int pc_overlap(int i, int c) {
  int d = i - 3 * c;
  return (d == 0 || d == 1) ? 4 : ((d == -1 || d == 2) ? 2 : 0);
}

// Packed ExperienceFrame (experience.py:10-18), 8 bytes:
//  byte0 x0 | y0<<4   state cell (before the action)
//  byte1 x1 | y1<<4   cell after the move -> with byte0 defines pixel_change
//  byte2 action       byte3 reward (int8)      byte4 bit0 terminal, bit7 valid
//  byte5 last_action  byte6 last_reward (int8) byte7 reserved (0)
UNREAL_HD uint64_t frame_pack(int x0, int y0, int x1, int y1, int action, int reward, int terminal,
                              int last_action, int last_reward) {
  uint64_t r = 0;
  r |= (uint64_t)((x0 & 15) | ((y0 & 15) << 4));
  r |= (uint64_t)((x1 & 15) | ((y1 & 15) << 4)) << 8;
  r |= (uint64_t)(action & 255) << 16;
  r |= (uint64_t)((uint8_t)(int8_t)reward) << 24;
  r |= (uint64_t)((terminal ? 1 : 0) | 0x80) << 32;
  r |= (uint64_t)(last_action & 255) << 40;
  r |= (uint64_t)((uint8_t)(int8_t)last_reward) << 48;
  return r;
}
// the record of a generic-frame env step (no cells): rewards stored as their sign
UNREAL_HD uint64_t framed_record(int action, float reward, int terminal, int last_action, float last_reward) {
  return frame_pack(0, 0, 0, 0, action, (reward > 0.f) - (reward < 0.f), terminal, last_action,
                    (last_reward > 0.f) - (last_reward < 0.f));
}
UNREAL_HD int frame_valid(uint64_t r) { return (int)((r >> 39) & 1); }
UNREAL_HD int frame_terminal(uint64_t r) { return (int)((r >> 32) & 1); }
UNREAL_HD int frame_reward(uint64_t r) { return (int)(int8_t)((r >> 24) & 255); }
UNREAL_HD int frame_last_reward(uint64_t r) { return (int)(int8_t)((r >> 48) & 255); }
UNREAL_HD int frame_action(uint64_t r) { return (int)((r >> 16) & 255); }
UNREAL_HD int frame_last_action(uint64_t r) { return (int)((r >> 40) & 255); }
UNREAL_HD int frame_x0(uint64_t r) { return (int)(r & 15); }
UNREAL_HD int frame_y0(uint64_t r) { return (int)((r >> 4) & 15); }
UNREAL_HD int frame_x1(uint64_t r) { return (int)((r >> 8) & 15); }
UNREAL_HD int frame_y1(uint64_t r) { return (int)((r >> 12) & 15); }

}  // namespace unreal
