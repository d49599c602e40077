from .agent_pool import DeviceAgentPool
from .cross_play import cross_play_returns

__all__ = ["DeviceAgentPool", "cross_play_returns"]
