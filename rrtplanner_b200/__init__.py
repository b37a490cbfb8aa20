"""rrtplanner_b200 -- B200-native tree-expansion hot path behind rrtplanner's planner API.

Drop-in for the classes of the reference's ``rrtplanner/rrt.py``::

    from rrtplanner_b200 import RRTStar, perlin_occupancygrid, random_point_og
    og = perlin_occupancygrid(512, 512)
    T, gv = RRTStar(og, n=5000, r_rewire=50).plan(random_point_og(og), random_point_og(og))

Importing the package does not need a GPU; the first kernel-backed call does (there is no CPU
fallback).  Build the CUDA library once with ``python -m rrtplanner_b200.build``.
"""
from . import worlds  # noqa: F401
from .worlds import perlin_occupancygrid  # noqa: F401
from .rrt import RRT, RRTStandard, RRTStar, RRTStarInformed, r2norm, random_point_og  # noqa: F401
from .dubins import RRTDubins, RRTStarDubins, dubins_collisionfree, dubins_length, dubins_path, dubins_points  # noqa: F401
from .body import body_layer, body_runs, car_body  # noqa: F401
from .batch import Batch2Result, BatchResult, DeviceBatch, DeviceBatch2, plan_batch, shard, shortcut_paths  # noqa: F401

__version__ = "0.1.0"
