"""clientCFD.draw() accumulation (clientCFD.pde:35-55) around a solver step of the CPU oracle, with the cadence of one
rlfc_env_step call for one environment.  The step is AFCCylinder.update() (`update_adaptive`, dt = checkCFL before
every step) by default; `update2` gives the fixed-dt step of ora_driver_step.  Float arithmetic is np.float32, one
rounding per operation, in the order of ora_driver_step.  Test infrastructure only."""
from __future__ import annotations

import numpy as np

f32 = np.float32


class DrawDriver:
    def __init__(self, env, substeps=16, resolution=24, init_time=1.0, episode_time=50.0, action_scale=5.0, adaptive=True):
        self.env = env
        self.substeps = int(substeps)
        self.resolution = int(resolution)
        self.init_time = f32(init_time)
        self.episode_time = f32(episode_time)
        self.adaptive = adaptive
        self.callLearn, self.Cd, self.Cl = self.substeps, f32(0), f32(0)
        self.obs = (f32(0), f32(0))
        self.solver_steps = 0

    @property
    def t(self):
        return f32(self.env.t)

    def _solver_step(self):
        """One solver step + the draw() accumulation; True when an observation was produced."""
        if self.adaptive:
            self.env.update_adaptive()
        else:
            self.env.update2()
        self.solver_steps += 1
        if not self.t > self.init_time:
            return False
        fx, fy = self.env.force()
        self.callLearn -= 1
        self.Cd = f32(self.Cd + fx)
        self.Cl = f32(self.Cl + fy)
        if self.callLearn <= 0:
            self.callLearn = self.substeps
            cl, two, res = f32(self.callLearn), f32(2), f32(self.resolution)
            self.Cd = f32(f32(f32(self.Cd / cl) * two) / res)
            self.Cl = f32(f32(f32(self.Cl / cl) * two) / res)
            self.obs = (self.Cl, self.Cd)
            return True
        return False

    def rl_step(self, action):
        """One rlfc_env_step for this environment: the action is taken only at a callLearn boundary past init_time; the
        environment then runs to its next observation, or until its episode is over.  Returns (obs, done)."""
        if self.t >= self.episode_time:
            return self.obs, True
        if self.t > self.init_time and self.callLearn == self.substeps:
            self.env.set_xi(*action)
        while True:
            produced = self._solver_step()
            if self.t >= self.episode_time or produced:
                break
        return self.obs, bool(self.t >= self.episode_time)
