// Part of the instantiation table of the register-resident trajectory kernels (see jq_traj_kernels.cuh): segment sweeps with the
// history VJP's paths (HIST = true, jq_seg_vjp_launch with a history or cotangent jumps), twins of the boundary-to-boundary sweeps of
// jq_traj_inst_e.cu (not the weighted tiles, which serve the propagator launch alone) and of jq_traj_inst_f.cu.
#include "jq_traj_kernels.cuh"

template <int NC, int NT, int JT = 0, int GLT = 0>
constexpr Inst tile_hist() { return traj_inst<TileLane<NC, NT>, 1, 1, JT, 0, GLT, TRAJ_WARPS, 0, true, true>(); }
template <int R, int NC, int UPL, int JT = 0, int GLT = 0, int OBJ = 0>
constexpr Inst fiber_hist() { return traj_inst<FiberLane<R, NC, 1>, UPL, 1, JT, OBJ, GLT, TRAJ_WARPS, 0, true, true>(); }

const Inst kInst[] = {
    tile_hist<2, 0, 4, 32>(), tile_hist<2, 0>(), tile_hist<3, 1, 3, 32>(), tile_hist<3, 1>(),
    fiber_hist<4, 1, 2, 5, 3>(), fiber_hist<4, 1, 2>(), fiber_hist<4, 1, 1>(), fiber_hist<6, 1, 2, 3, 4>(), fiber_hist<6, 1, 2>(),
    fiber_hist<3, 1, 1>(), fiber_hist<3, 1, 2>(), fiber_hist<5, 1, 2>(), fiber_hist<2, 1, 1>(),
    fiber_hist<4, 2, 1>(), fiber_hist<3, 2, 1>(), fiber_hist<4, 3, 1>(), fiber_hist<3, 3, 1>(),
    // the gradient sweep (mode 5) with the jumps in the second adjoint set
    fiber_hist<3, 2, 1, 0, 0, 1>(), fiber_hist<4, 2, 1, 0, 0, 1>(), fiber_hist<4, 1, 1, 0, 0, 1>(), fiber_hist<4, 1, 2, 0, 0, 1>(),
    fiber_hist<6, 1, 2, 0, 0, 1>(), fiber_hist<4, 3, 1, 0, 0, 1>(), fiber_hist<2, 1, 1, 0, 0, 1>(),
};
const InstPart kInstG = inst_part(kInst);
