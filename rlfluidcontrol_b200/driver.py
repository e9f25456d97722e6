"""Batched episode driver: the loop of clientLilypad/clientCFD.pde for B environments at once.

The reference client (clientCFD.pde:18-133) owns ONE environment: init -> start_episode -> [update2 ... every 16 solver
steps after t > initTime: request_stochastic_action("<Cl>_<Cd>")] -> at t >= Time: train(1000), save(1000), new sim.  This
driver keeps that order per environment on top of the C ABI (`rlfc_env_step`, which advances every environment to its next
observation) and talks to the agent through ONE `request_batch_action` call per RL step (the peer's protocol extension,
rlfluidcontrol_b200/peer/agent_server.py; the unchanged single-environment protocol is served by csrc/rlfc_client.c):

  * observations travel as Java-formatted decimal text, "<Cl>_<Cd>" per environment joined by ';', exactly what
    clientCFD.pde:119 builds for one environment; actions come back as "<a1>_<a2>" and are parsed like Float.parseFloat;
  * a failed RPC leaves the actions at (0, 0) (clientCFD.pde:118-132);
  * an environment whose episode is over (t >= Time) is reset on its own (`auto-reset`): its record stream is closed on
    the peer (`finish_envs`), it restarts from the init state with xi = 0 and -- like the sketch globals callLearn/Cd/Cl
    (clientCFD.pde:11-13) -- keeps its force accumulators unless `reset_accumulators` is set.  Its first observation after
    the reset comes out of the uncontrolled start (rlfc.h: rlfc_env_step), during which the others wait;
  * after every `train_every` finished environment-episodes: train(train_steps), save(train_steps) (clientCFD.pde:72-81);
  * `sample_params` (a handle created with env_params): setUpNewSim builds a new AFCCylinder (clientCFD.pde:93-102), so a
    finished environment may start its next episode with new constructor arguments: sample_params(rng, env_ids) returns
    one parameter set per finished environment (dicts or a structured array, see AFCCylinderBatch.reset).
"""
from __future__ import annotations

import ctypes as C
import xmlrpc.client

import numpy as np


class BatchedEpisodeDriver:
    def __init__(self, env, url="http://localhost:8000", train_steps=1000, train_every=None, reset_accumulators=False,
                 proxy=None, quiet=True, sample_params=None, seed=None):
        self.env = env
        self.B = env.n_envs
        self.peer = proxy if proxy is not None else xmlrpc.client.ServerProxy(url, allow_none=True)
        self.train_steps = train_steps
        self.train_every = train_every if train_every is not None else self.B
        self.reset_accumulators = reset_accumulators
        self.quiet = quiet
        self.sample_params = sample_params
        self.rng = np.random.default_rng(seed)
        self.finished_episodes = 0
        self.rl_steps = 0
        self.episode_returns = []
        self._ret = np.zeros(self.B, np.float64)
        L = env._L
        L.rlfc_format_float_java.argtypes = [C.c_float, C.c_char_p, C.c_int]
        self._fmt_buf = C.create_string_buffer(64)
        self._L = L

    # String.valueOf(float) of the reference (clientCFD.pde:119)
    def _jf(self, v):
        self._L.rlfc_format_float_java(float(v), self._fmt_buf, 64)
        return self._fmt_buf.value.decode()

    def _rpc(self, name, arg, default):
        try:
            return getattr(self.peer, name)(arg)
        except Exception as exc:                      # clientCFD.pde:20-29,122-130: print and carry on
            if not self.quiet:
                print(f"{name}: RPC failed ({exc})")
            return default

    def start(self):
        """setup() + setUpNewSim(): init(-1), start_episode(-1), then the uncontrolled start of every environment."""
        self._rpc("init", -1, False)
        self._rpc("start_episode", -1, True)
        self.env.reset(reset_accumulators=True)
        self.obs, _, self.done = self.env.step(np.zeros((self.B, 2), np.float32))
        self._has_obs = np.ones(self.B, bool)
        return self.obs

    def _ask(self):
        payload = ";".join(f"{self._jf(o[0])}_{self._jf(o[1])}" if h else "" for o, h in zip(self.obs, self._has_obs))
        reply = self._rpc("request_batch_action", payload, None)
        acts = np.zeros((self.B, 2), np.float32)      # zeros on failure
        if isinstance(reply, str):
            parts = reply.split(";")
            if len(parts) == self.B:
                for e, p in enumerate(parts):
                    try:
                        a1, a2 = p.split("_")
                        acts[e] = (np.float32(a1), np.float32(a2))
                    except ValueError:
                        pass
        return acts

    def step(self):
        """One RL step of the whole batch: ask, act, observe; finished environments are reset for the next call."""
        acts = self._ask()
        self.obs, rew, self.done = self.env.step(acts)
        self._ret += rew
        self.rl_steps += 1
        self._has_obs[:] = True
        fin = np.flatnonzero(self.done)
        if len(fin):
            self._rpc("finish_envs", ";".join(str(int(e)) for e in fin), True)
            for e in fin:
                self.episode_returns.append(float(self._ret[e]))
                self._ret[e] = 0
            before = self.finished_episodes // self.train_every
            self.finished_episodes += len(fin)
            if self.finished_episodes // self.train_every > before:      # clientCFD.pde:72-81
                self._rpc("train", self.train_steps, True)
                self._rpc("save", self.train_steps, True)
            params = None if self.sample_params is None else self.sample_params(self.rng, fin)
            self.env.reset(fin, reset_accumulators=self.reset_accumulators, params=params)
            # the reset environments produce their first observation during the next env.step (uncontrolled start,
            # actions ignored); what they hold now is the previous episode's last observation: not sent to the agent
            self._has_obs[fin] = False
        return self.obs, rew, self.done

    def run(self, rl_steps):
        self.start()
        for _ in range(rl_steps):
            self.step()
        return self
