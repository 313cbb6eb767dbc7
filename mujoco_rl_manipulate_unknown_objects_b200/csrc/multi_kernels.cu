// The mixed-simulator (several scenes, SimBuffers::nobj > 1) instantiations of the per-environment kernels, in a translation unit of
// their own so that the single-scene kernels of gripper_sim.cu keep stage functions specialised to one constant model address
// (env_lockstep.cuh : SimKernels).
#include "env_lockstep.cuh"

namespace grs {
SimKernels multi_sim_kernels() { return sim_kernels<true>(); }
}  // namespace grs
