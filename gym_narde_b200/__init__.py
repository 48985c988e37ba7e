"""gym_narde_b200 -- B200-native batched Narde environment (drop-in for gym_narde's env path).

Public surface (mirrors gym_narde/__init__.py + gym_narde/envs):
  gym_narde_b200.envs.NardeEnv / Narde   single-game facade, same names as the reference
  gym_narde_b200.VecNardeEnv             N lock-step games on the GPU
  gym_narde_b200.AfterstateMLP / AfterstateActor   DecomposedDQN(198) scorer and the greedy batched actor
  gym_narde_b200.LookaheadActor          the same actor with a one-ply expectimax over the opponent's 21 rolls
  gym_narde_b200.AfterstateMatch         lock-step games of two afterstate nets, or a net and the random agent, tallied
                                         on the device
  gym_narde_b200.expand_obs198(lo, hi)   packed 32-byte state records -> Box(198) rows (host or device)
  gym_narde_b200.NardeGameManager        interactive turn manager (my_game/narde_game_manager.py surface)
  gym_narde_b200.make(id)                'narde-v0' (reference rules) / 'Narde-v0' (README rules)
When gymnasium is importable both ids are also registered with it (max_episode_steps=1000, as
gym_narde/__init__.py:3-7 does).
"""
__version__ = "0.1.0"


def _lazy(name):
    if name == "VecNardeEnv":
        from .vec_env import VecNardeEnv
        return VecNardeEnv
    if name == "NardeEnv":
        from .envs.narde_env import NardeEnv
        return NardeEnv
    if name == "Narde":
        from .envs.narde import Narde
        return Narde
    if name == "AfterstateMLP":
        from .mlp import AfterstateMLP
        return AfterstateMLP
    if name == "AfterstateActor":
        from .actor import AfterstateActor
        return AfterstateActor
    if name == "LookaheadActor":
        from .lookahead import LookaheadActor
        return LookaheadActor
    if name == "AfterstateMatch":
        from .match import AfterstateMatch
        return AfterstateMatch
    if name == "expand_obs198":
        from .state import expand_obs198
        return expand_obs198
    if name == "NardeGameManager":
        from .narde_game_manager import NardeGameManager
        return NardeGameManager
    raise AttributeError(name)


def __getattr__(name):
    return _lazy(name)


class TimeLimit:
    """gymnasium's TimeLimit for the make() fallback below: truncated=True once max_episode_steps steps were taken
    since the last reset (the wrapper gym.make applies for gym_narde/__init__.py:6 `max_episode_steps=1000`)."""

    def __init__(self, env, max_episode_steps):
        self.env = env
        self._max_episode_steps = int(max_episode_steps)
        self._elapsed_steps = 0

    @property
    def unwrapped(self):
        return self.env.unwrapped

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        return getattr(self.env, name)

    def reset(self, **kwargs):
        self._elapsed_steps = 0
        return self.env.reset(**kwargs)

    def step(self, action):
        obs, reward, terminated, truncated, info = self.env.step(action)
        self._elapsed_steps += 1
        if self._elapsed_steps >= self._max_episode_steps:
            truncated = True
        return obs, reward, terminated, truncated, info

    def render(self):
        return self.env.render()

    def close(self):
        return self.env.close()


MAX_EPISODE_STEPS = 1000  # gym_narde/__init__.py:6


def make(env_id="narde-v0", max_episode_steps=MAX_EPISODE_STEPS, **kwargs):
    """gym.make('gym_narde:narde-v0') without gymnasium: the env wrapped in the TimeLimit the registration implies
    (max_episode_steps=None or 0: no wrapper)."""
    from .envs.narde_env import NardeEnv

    base = env_id.split(":")[-1]
    if base == "narde-v0":
        env = NardeEnv(rules="reference", **kwargs)
    elif base == "Narde-v0":
        env = NardeEnv(rules="full", **kwargs)
    else:
        raise ValueError("unknown env id %r" % env_id)
    return TimeLimit(env, max_episode_steps) if max_episode_steps else env


def _register_with_gymnasium():
    """gym_narde/__init__.py:3-7 for both ids; a no-op without gymnasium."""
    try:
        from gymnasium.envs.registration import register as _register
    except ImportError:
        return False
    _register(id="narde-v0", entry_point="gym_narde_b200.envs:NardeEnv", max_episode_steps=MAX_EPISODE_STEPS)
    _register(id="Narde-v0", entry_point="gym_narde_b200.envs:NardeEnv", max_episode_steps=MAX_EPISODE_STEPS,
              kwargs={"rules": "full"})
    return True


_register_with_gymnasium()
