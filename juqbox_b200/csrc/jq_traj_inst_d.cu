// Part of the instantiation table of the register-resident trajectory kernels (see jq_traj_kernels.cuh): tile layout.
#include "jq_traj_kernels.cuh"

const Inst kInst[] = {
    traj_inst<TileLane<2, 2>, 1, 1, 4, 0, 16>(),            // cnot2 example shape: 4 x 4 levels, 2 x 2 tiles, J = 4, 16-lane groups (two trajectories per warp)
    traj_inst<TileLane<2, 1, 1>, 1, 2, 4, 0, 8>(),          // the same, first subsystem whole in the lane: 8 elements per lane, 8-lane groups (four trajectories per warp)
    traj_inst<TileLane<2, 2>, 1>(),                          // 4 x 4 levels, run-time J and group size
    traj_inst<TileLane<3, 3>, 1, 1, 3, 0, 32, 8>(),         // cnot3 example shape: 4 x 4 x 4 levels, 2 x 2 x 2 tiles (one warp per trajectory), J = 3, 8 warps per CTA
    traj_inst<TileLane<3, 3>, 1, 1, 0, 0, 0, 8>(),          // 4 x 4 x 4 levels, run-time J and group size
    // latency layout for small batches (kernel id 5), with pipelined state / adjoint roles: one element per lane, 64 lanes per
    // 4 x 4 x 4-column trajectory
    traj_inst<TileLane<2, 0>, 1, 1, 4, 0, 32, 2, 1>(), traj_inst<TileLane<2, 0>, 1, 1, 0, 0, 0, 2, 1>(),
    // 4 x 4 x 4 levels: first subsystem in halves, 2 elements per lane, one warp per column; state + adjoint share a role (register budget)
    traj_inst<TileLane<3, 1>, 1, 1, 3, 0, 32, 4, 2>(), traj_inst<TileLane<3, 1>, 1, 1, 0, 0, 0, 4, 2>(),
    // single-fibre layout, pipelined roles: single qudits, risk-neutral SWAP 0-2 (J = 5) and n = 4, cnot1 (n = 6), rabi (n = 2)
    traj_inst<FiberLane<4, 1, 1>, 2, 1, 5, 0, 3, 1, 1>(), traj_inst<FiberLane<4, 1, 1>, 2, 1, 0, 0, 0, 1, 1>(), traj_inst<FiberLane<4, 1, 1>, 1, 1, 0, 0, 0, 1, 1>(),
    traj_inst<FiberLane<6, 1, 1>, 2, 1, 3, 0, 4, 1, 1>(), traj_inst<FiberLane<6, 1, 1>, 2, 1, 0, 0, 0, 1, 1>(), traj_inst<FiberLane<2, 1, 1>, 1, 1, 0, 0, 0, 1, 1>(),
};
const InstPart kInstD = inst_part(kInst);
