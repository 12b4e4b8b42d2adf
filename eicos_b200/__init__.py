"""eicos_b200 - B200-native batched SOCP interior-point engine behind EiCOS's solver API.

Only the hot path of EmbersArc/EiCOS is here (Solver construction -> solve -> updateData ->
solution, plus a batched overload); see DESIGN.md.  The compute path is hand-written CUDA for
sm_100a in eicos_b200/csrc, reached through the C ABI in include/eicos_b200.h.
"""
from .binding import BatchSolver, Library, MultiBatchSolver, Settings, Solver, default_settings, load, PRODUCT_LIB, EXPORTS  # noqa: F401
