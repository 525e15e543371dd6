from .policy import PolicyBase
from .mpc_policy import MpcPolicy
from .cem_mpc import CemMpc
from .safe_cem_mpc import SafeCemMpc
from .mppi_mpc import MppiMpc, SafeMppiMpc
from .random_shooting_mpc import RandomShootingMpc, RandomMpc
