"""CPU checks of the draw() driver the adaptive-dt RL-step tests compare against (tests/adaptive_driver.py)."""
import numpy as np

from adaptive_driver import DrawDriver
from conftest import config1_actions


def _oracle_env(oracle, init_state):
    e = oracle.OracleEnv(literal=False)
    e.set_state(init_state["ux"], init_state["uy"], init_state["p"])
    return e


def test_fixed_dt_driver_matches_oracle_driver(oracle, init_state):
    """With the fixed-dt step the driver reproduces ora_driver_step (OracleEnv.env_step) exactly."""
    ref = _oracle_env(oracle, init_state)
    drv = DrawDriver(_oracle_env(oracle, init_state), init_time=-1.0, adaptive=False)
    for k in range(2):
        a = config1_actions(k)
        o_ref = ref.env_step(a)
        o, done = drv.rl_step(a)
        assert (o[0], o[1]) == (np.float32(o_ref[0]), np.float32(o_ref[1])) and not done
    assert drv.t == np.float32(ref.t) and drv.solver_steps == 32


def test_adaptive_driver_cadence(oracle, init_state):
    """Adaptive steps: the first call runs uncontrolled past init_time and then one accumulation window; the episode
    ends where t crosses episode_time, and later calls take no step."""
    drv = DrawDriver(_oracle_env(oracle, init_state), init_time=0.05, episode_time=0.6)
    o, done = drv.rl_step((0.5, -0.5))
    assert not done and drv.callLearn == 16 and drv.t > np.float32(0.05)
    n0 = drv.solver_steps
    assert n0 > 16
    while not done:
        o, done = drv.rl_step((0.5, -0.5))
    assert drv.t >= np.float32(0.6)
    n1 = drv.solver_steps
    assert drv.rl_step((0.0, 0.0)) == (o, True) and drv.solver_steps == n1
    assert 0 < drv.env.dt <= 1
