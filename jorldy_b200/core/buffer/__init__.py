from .rollout_buffer import RolloutBuffer, DeviceRollout  # noqa: F401
from .replay_buffer import ReplayBuffer  # noqa: F401
from .per_buffer import PERBuffer  # noqa: F401
from .frame_replay import FrameReplayBuffer, FramePERBuffer  # noqa: F401
