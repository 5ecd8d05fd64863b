"""Batched on-policy rollout + targets engine: the device side of Trainer._process_base's
environment loop and reverse scans (train/trainer.py:218-336) and of the pixel-control
target scan (trainer.py:352-372) for N mazes at once.

One *pass* = K1 (step + render + pixel-change of all T rollout steps: one window launch, or
T launches each writing its own [t] slice of the rollout buffers) followed by ONE targets
launch (unreal_maze_rollout_targets: n-step returns, advantages and PC Q-targets from the
frame records K1 wrote; the pixel-change maps are not read back).  The two phases are
captured into CUDA graphs, so a pass costs two graph launches.  All rollout buffers stay
resident in HBM for the learner:

  obs      [T, N, 84, 84, 3]  f32 | u8     model input of each step's *next* state
  pc       [T, N, 20, 20]     f32          pixel change caused by each step
  reward   [T, N] f32, terminal [T, N] u8
  R, adv   [T, N] f32                      n-step returns / advantages
  pc_tgt   [T, N, 20, 20]     f32          pixel-control Q targets
"""
import torch

from .. import _lib
from .. import kernels as K


class RolloutTargets(object):
  def __init__(self, num_envs, rollout_len=20, gamma=0.99, gamma_pc=0.9, obs_dtype=torch.float32,
               device="cuda:0", auto_reset=True, use_graphs=True, window_kernel=None):
    self.n = int(num_envs)
    self.t = int(rollout_len)
    self.gamma = float(gamma)
    self.gamma_pc = float(gamma_pc)
    self.device = torch.device(device)
    self.auto_reset = auto_reset
    self.use_graphs = use_graphs
    # the T actions of a pass are inputs, so all T steps go out as ONE launch (unreal_maze_window) instead of T K1
    # launches: no launch ramps / drains between the steps (f32: 7.1 TB/s instead of 6.45; u8: the ramp was a third of
    # a 14 us transfer).  Same results either way (tests/test_gpu_rollout_bench_config.py); False = one launch per step,
    # which is what a rollout whose actions depend on the observations (Trainer) has to do.
    self.window_kernel = (self.t <= 32) if window_kernel is None else bool(window_kernel)
    if self.window_kernel and self.t > 32:
      raise _lib.UnrealError("the window kernel covers at most 32 rollout steps")
    d, n, t = self.device, self.n, self.t
    with torch.cuda.device(d):
      self.state = K.MazeState(n, d)
    # inputs of a pass (filled by the policy / value heads, or by the caller)
    self.actions = torch.zeros(t, n, dtype=torch.int32, device=d)
    self.values = torch.zeros(t, n, dtype=torch.float32, device=d)
    self.boot_value = torch.zeros(n, dtype=torch.float32, device=d)
    self.boot_q = torch.zeros(n, 20, 20, dtype=torch.float32, device=d)
    # outputs
    self.obs = torch.empty(t, n, 84, 84, 3, dtype=obs_dtype, device=d)
    self.pc = torch.empty(t, n, 20, 20, dtype=torch.float32, device=d)
    self.reward = torch.empty(t, n, dtype=torch.float32, device=d)
    self.terminal = torch.empty(t, n, dtype=torch.uint8, device=d)
    self.frame_rec = torch.empty(t, n, dtype=torch.int64, device=d)
    self.R = torch.empty(t, n, dtype=torch.float32, device=d)
    self.adv = torch.empty(t, n, dtype=torch.float32, device=d)
    self.pc_tgt = torch.empty(t, n, 20, 20, dtype=torch.float32, device=d)
    self._graphs = None
    # host staging for the host-buffer entry point (pinned, reused every pass)
    self._h_in = None
    self._h_out = None
    self._copy_stream = None
    self.host_graph = True       # run_host(): the copies + phases as one CUDA graph (False: ~15 stream calls per pass)
    self._host_graph = None

  # launches per pass, by kernel
  @property
  def launches_per_pass(self):
    # window form: u8 = one warp-per-env kernel; f32 = one CTA-per-item kernel + the state kernel; + the targets kernel
    return ((1 if self.obs.dtype == torch.uint8 else 2) if self.window_kernel else self.t) + 1

  # ---- the two phases, eager ----------------------------------------------------------
  def _steps(self):
    if self.window_kernel:
      K.maze_window(self.state, self.actions, obs=self.obs, pc=self.pc, reward=self.reward, terminal=self.terminal,
                    frame_rec=self.frame_rec, auto_reset=self.auto_reset)
      return
    for t in range(self.t):
      K.maze_step(self.state, self.actions[t], obs=self.obs[t], pc=self.pc[t], reward=self.reward[t],
                  terminal=self.terminal[t], frame_rec=self.frame_rec[t], auto_reset=self.auto_reset)

  def _targets(self):
    K.maze_rollout_targets(self.frame_rec, self.values, self.boot_value, self.boot_q, self.gamma, self.gamma_pc,
                           self.R, self.adv, self.pc_tgt)

  def _capture(self):
    torch.cuda.synchronize(self.device)
    self._steps(); self._targets()                            # warm the lazy init paths before capture
    K.maze_reset(self.state)
    torch.cuda.synchronize(self.device)
    graphs = []
    for fn in (self._steps, self._targets):
      g = torch.cuda.CUDAGraph()
      with _lib.graph_capture(g):
        fn()
      graphs.append(g)
    self._graphs = graphs

  def run_device(self, events=None):
    """One pass with inputs already in HBM.  `events`: optional list of 4 CUDA events recorded
    on the current stream before K1 / after K1 / after the targets launch / again after it (the
    targets of K3 and K4 are one launch; the fourth event keeps the K1 / K3 / K4 timing layout,
    with a K4 span of ~0)."""
    with torch.cuda.device(self.device):
      if self.use_graphs and self._graphs is None:
        self._capture()
      phases = [g.replay for g in self._graphs] if self.use_graphs else [self._steps, self._targets]
      if events is not None:
        events[0].record()
      for i, ph in enumerate(phases):
        ph()
        if events is not None:
          events[i + 1].record()
      if events is not None:
        events[3].record()

  # ---- host-buffer entry point (what a CPU-side caller of the reference API would use) --
  def _ensure_host(self):
    if self._h_in is None:
      t, n = self.t, self.n
      pin = dict(pin_memory=True)
      self._h_in = dict(actions=torch.zeros(t, n, dtype=torch.int32, **pin),
                        values=torch.zeros(t, n, dtype=torch.float32, **pin),
                        boot_value=torch.zeros(n, dtype=torch.float32, **pin),
                        boot_q=torch.zeros(n, 20, 20, dtype=torch.float32, **pin))
      self._h_out = dict(reward=torch.zeros(t, n, dtype=torch.float32, **pin),
                         terminal=torch.zeros(t, n, dtype=torch.uint8, **pin),
                         R=torch.zeros(t, n, dtype=torch.float32, **pin),
                         adv=torch.zeros(t, n, dtype=torch.float32, **pin))

  @property
  def h2d_bytes_per_pass(self):
    self._ensure_host()
    return sum(v.numel() * v.element_size() for v in self._h_in.values())

  @property
  def d2h_bytes_per_pass(self):
    self._ensure_host()
    return sum(v.numel() * v.element_size() for v in self._h_out.values())

  def host_inputs(self):
    """Pinned host staging buffers (numpy views) a caller can fill in place: actions [T,N] i32,
    values [T,N] f32, boot_value [N] f32, boot_q [N,20,20] f32.  Passing these same arrays (or
    None) to run_host() skips the host-side staging copy."""
    self._ensure_host()
    return {k: v.numpy() for k, v in self._h_in.items()}

  def run_host(self, actions=None, values=None, boot_value=None, boot_q=None):
    """One pass from HOST buffers (numpy or CPU tensors): copies the inputs host->device,
    runs the pass, copies rewards / terminals / returns / advantages back and returns them
    as numpy views of pinned memory (valid until the next call).  Frames, pixel-change maps
    and PC targets stay on the device for the learner.

    The copies are pipelined around the two phases on a second stream: only the actions
    (T*N*4 bytes) gate K1; values / bootstraps travel while K1 runs and are waited for just
    before the targets launch, rewards / terminals return under the targets kernel and
    returns / advantages after it."""
    self._ensure_host()
    hi, ho = self._h_in, self._h_out
    for name, arr in (("actions", actions), ("values", values), ("boot_value", boot_value), ("boot_q", boot_q)):
      if arr is None:
        continue
      t = torch.as_tensor(arr)
      if t.data_ptr() != hi[name].data_ptr():       # not already the pinned staging buffer
        hi[name].copy_(t)
    with torch.cuda.device(self.device):
      if self.use_graphs and self._graphs is None:
        self._capture()
      if self._copy_stream is None:
        self._copy_stream = torch.cuda.Stream(self.device)
        self._ev = [torch.cuda.Event() for _ in range(5)]
      main = torch.cuda.current_stream()
      if self.use_graphs and self.host_graph:
        # the whole pass -- the H2D copies, the two phases and the D2H copies with their cross-stream overlap -- as ONE
        # CUDA graph over the pinned staging buffers: one launch and one synchronisation per call instead of ~15 API calls
        if self._host_graph is None:
          self._pipeline(main)                                # THIS call's pass, eagerly (creates every lazy resource)
          main.synchronize()
          g = torch.cuda.CUDAGraph()
          with _lib.graph_capture(g):                         # recorded for the following calls, not executed
            self._pipeline(torch.cuda.current_stream(), replay_graphs=False)
          self._host_graph = g
        else:
          self._host_graph.replay()
      else:
        self._pipeline(main)
      main.synchronize()
    return {k: v.numpy() for k, v in self._h_out.items()}

  def _pipeline(self, main, replay_graphs=True):
    """The copies and phases of one host-buffer pass on `main` + the copy stream (see run_host)."""
    hi, ho = self._h_in, self._h_out
    side = self._copy_stream
    ev_start, ev_in, ev_k1, ev_tg, ev_out = self._ev
    phases = ([g.replay for g in self._graphs] if (self.use_graphs and replay_graphs)
              else [self._steps, self._targets])
    ev_start.record(main)
    self.actions.copy_(hi["actions"], non_blocking=True)
    side.wait_event(ev_start)                      # previous pass has finished with the inputs
    with torch.cuda.stream(side):
      self.values.copy_(hi["values"], non_blocking=True)
      self.boot_value.copy_(hi["boot_value"], non_blocking=True)
      self.boot_q.copy_(hi["boot_q"], non_blocking=True)
      ev_in.record(side)
    phases[0]()                                    # K1 (window kernel, or T launches)
    ev_k1.record(main)
    with torch.cuda.stream(side):
      side.wait_event(ev_k1)
      ho["reward"].copy_(self.reward, non_blocking=True)
      ho["terminal"].copy_(self.terminal, non_blocking=True)
    main.wait_event(ev_in)
    phases[1]()                                    # targets: R, adv, PC targets
    ev_tg.record(main)
    with torch.cuda.stream(side):
      side.wait_event(ev_tg)
      ho["R"].copy_(self.R, non_blocking=True)
      ho["adv"].copy_(self.adv, non_blocking=True)
      ev_out.record(side)
    main.wait_event(ev_out)
