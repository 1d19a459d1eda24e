"""motionplanning.jl_b200 -- B200-native back-end for the data-parallel hot path of
schmrlng/MotionPlanning.jl (importable as `mpb200` through the shim at the repository root).

Host-side mirror of the reference's plug-in interface (same names, argument meaning and error
behaviour) above the C ABI of libmpb200.so (include/mpb200.h).  All compute happens in
hand-written sm_100a CUDA kernels; there is no CPU fallback.
"""
from ._lib import MPB200Error, init, load  # noqa: F401
from .shapes2d import Box2D, Circle, Compound2D, Polygon, Shape2D  # noqa: F401
from .collisioncheckers import (BoxBounds, CollisionChecker, PointRobot2D, PointRobotNDBoxes,  # noqa: F401
                                SweptCollisionChecker, addblocker, addobstacle, inflate)
from .statespaces import (BoundedEuclideanStateSpace, BoundedStateSpace, Euclidean, Identity,  # noqa: F401
                          OutputMatrix, UnitHypercube, VectorView, dim, is_free_motion, is_free_path,
                          is_free_state, segments_free, state2workspace, states_free, volume)
from .nearneighbors import (ImmutableNNC, MetricNN, QuasiMetricNN, SampleSet, SparseMatrixCSC, SparseVectorView,  # noqa: F401
                            loadNN, saveNN,
                            addpoints, filter_neighborhood, inball, inballB, inballF, nonzeroinds,
                            nonzeros, viewcol, knn, knnB, knnF, mutualknn, mutualknnF)
from .linearquadratic import (DoubleIntegrator, LinearQuadratic, LinearQuadraticQuasiMetricSpace,  # noqa: F401
                              lq_motions_free, setup_steering, steer, steer_batch)
from .simplecars import (ChoppedMetric, ChoppedQuasiMetric, DubinsExact, DubinsQuasiMetricSpace, ReedsSheppExact,  # noqa: F401
                         ReedsSheppMetricSpace, car_motions_free, car_steer_batch, steering_control)
from .problems import (BallGoal, MPProblem, MPSolution, PointGoal, RectangleGoal, StateGoal, is_goal_pt,  # noqa: F401
                       sample_free, sample_free_goal, sample_goal)
from .planners import fmtstar, gmtstar, gmtstar_batch, shortcut_paths  # noqa: F401
from . import montecarlo  # noqa: F401
from .montecarlo import MCProblem, collision_probability  # noqa: F401
from . import obstaclesets  # noqa: F401

__version__ = "0.1.0"
