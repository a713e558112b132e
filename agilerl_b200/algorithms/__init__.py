from .dqn import DQN
from .dqn_rainbow import RainbowDQN
from .maddpg import MADDPG
from .matd3 import MATD3
from .td3 import DDPG, TD3

__all__ = ["DQN", "RainbowDQN", "DDPG", "TD3", "MADDPG"]   # MATD3 is importable but not aliased by install() (see matd3.py)
