# SHMIP-like moulin run: 100 km x 20 km margin with the SHMIP square-root surface, a small background input and
# 60 seeded moulins with diurnal hydrographs (shakti_b200.configs.moulins_like).  The SHMIP moulin position files
# are not shipped, so the positions are seeded and the results are not SHMIP numbers.
from _synthetic import md_from_case
from shakti_b200 import configs


def initialize(comm):
    days = 5
    case = configs.moulins_like(nx=200, ny=40, nsteps=days * 24)
    md = md_from_case(comm, case, __file__, nt_save=6)
    md.moulins = case.meta["moulins"]            # (x, y, times, Q): snapped to the nearest mesh vertex
    md.moulin_period = case.meta["moulin_period"]
    return md
