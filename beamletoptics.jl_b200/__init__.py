"""beamletoptics.jl_b200 -- B200-native (sm_100a) trace hot path of BeamletOptics.jl.

Host-side mirror of the reference's API for the path `solve_system!` drives (System/ObjectGroup
construction, kinematics, Beam / GaussianBeamlet, Photodetector / Spotdetector); all per-ray work
runs in hand-written CUDA kernels behind the C ABI of include/bmo.h (libbmo.so).  Julia's `f!`
is spelled `f_` here.  There is no CPU fallback.
"""
from . import linalg
from ._lib import BmoError, counters, counters_reset, measure_fp64_peak
from .beams import (Beam, BeamletBundle, CollimatedSource, DeviceBeamletSource, DeviceSource, GaussianBeamlet, Intersection, PointSource, PolarizedRay, Ray,
                    RayBundle, UniformDiscSource)
from .components import (AcylindricalSurface, CircularFlatSurface, ConcaveSphericalMirror, CubeBeamsplitter, EvenAsphericalSurface, LensFromSurfaces, SphericalSurface, CylindricalLens, CylindricalSurface, RectangularFlatSurface, DiscreteRefractiveIndex, DoubletLens, IntersectableObject, Lens,
                         MeshDummy, Mirror, NonInteractableObject, ObjectGroup, PSFDetector, Photodetector, PolarizationFilter, Prism, RectangularCompensatorPlate,
                         RectangularPlanoMirror, RectangularPlateBeamsplitter, Retroreflector, RightAnglePrism, RightAnglePrismMirror,
                         RoundPlanoMirror, RoundPlateBeamsplitter, RoundThinBeamsplitter, SellmeierEquation, SphericalDoubletLens,
                         SphericalLens, Spotdetector, SquarePlanoMirror, SquarePlanoMirror2D, StaticSystem, System, ThinBeamsplitter,
                         ThinLens, XYBasis, XZBasis, YZBasis, inch, lens_shape)
from .shapes import (AcylindricalSurfaceSDF, AsphericalSurfaceSDF, BoxSDF, CircularFlatMesh, ConcaveAsphericalSurfaceSDF, ConvexAsphericalSurfaceSDF, ConcaveCylinderSDF, ConcaveSphericalSurfaceSDF, ConvexCylinderSDF, ConvexSphericalSurfaceSDF, CubeMesh, CuboidMesh, CutSphereSDF,
                     CylinderSDF, Mesh, MeniscusLensSDF, PlanoSurfaceSDF, QuadraticFlatMesh, RectangularFlatMesh, RetroMesh,
                     RightAnglePrismSDF, RingSDF, SphereSDF, ThinLensSDF, UnionSDF, load_stl)
from .solver import DeviceSystem, TraceResult, pd_accumulate, retrace, solve_system_, spot_stats, spot_stats_poses, trace_beamlets, trace_rays, trace_rays_spots, upload_system
from .sweep import (flatten_poses, solve_pose_sweep, KinProgram, get_pose_tables, solve_pose_sweep_device, solve_spot_sweep,
                    solve_spot_sweep_device, tile_ray_bundle)
from . import parallel
from .parallel import solve_pose_sweep_sharded, solve_spot_sharded, solve_spot_sweep_sharded, solve_system_sharded


# function-style kinematic API of the reference: translate3d!(obj, v) -> translate3d_(obj, v)
def translate3d_(obj, offset): obj.translate3d_(offset)
def translate_to3d_(obj, target): obj.translate_to3d_(target)
def rotate3d_(obj, axis, theta): obj.rotate3d_(axis, theta)
def xrotate3d_(obj, theta): obj.xrotate3d_(theta)
def yrotate3d_(obj, theta): obj.yrotate3d_(theta)
def zrotate3d_(obj, theta): obj.zrotate3d_(theta)
def align3d_(obj, axis): obj.align3d_(axis)
def reset_translation3d_(obj): obj.reset_translation3d_()
def reset_rotation3d_(obj): obj.reset_rotation3d_()
def position(obj): return obj.position()
def orientation(obj): return obj.orientation()
def thickness(obj): return obj.thickness()
def empty_(det): det.empty_()
def optical_power(pd): return pd.optical_power()
def intensity(pd): return pd.intensity()
