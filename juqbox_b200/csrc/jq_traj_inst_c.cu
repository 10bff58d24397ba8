// Part of the instantiation table of the register-resident trajectory kernels (see jq_traj_kernels.cuh).
#include "jq_traj_kernels.cuh"

const Inst kInst[] = {
    traj_inst<FiberLane<3, 2, 1>, 1, 1, 0, 1>(), traj_inst<FiberLane<4, 2, 1>, 1, 1, 0, 1>(), traj_inst<FiberLane<4, 1, 1>, 1, 1, 0, 1>(),   // objFuncType 2/3
    traj_inst<FiberLane<4, 1, 1>, 2, 1, 0, 1>(), traj_inst<FiberLane<6, 1, 1>, 2, 1, 0, 1>(), traj_inst<FiberLane<4, 3, 1>, 1, 1, 0, 1>(),
    traj_inst<FiberLane<2, 1, 1>, 1, 1, 0, 1>(),
    // drift with exchange couplings to the fibre subsystem (HX: every control outside LMASK)
    traj_inst<FiberLane<4, 2, 1, 1, 0, 2>, 1>(), traj_inst<FiberLane<3, 2, 1, 1, 0, 2>, 1>(), traj_inst<FiberLane<2, 2, 1, 1, 0, 2>, 1>(), traj_inst<FiberLane<4, 3, 1, 1, 0, 6>, 1>(),
    traj_inst<FiberLane<3, 2, 1>, 1, 1, -1>(), traj_inst<FiberLane<4, 2, 1>, 1, 1, -1>(), traj_inst<FiberLane<4, 1, 1>, 2, 1, -1>(),      // Jacobi solver
    traj_inst<FiberLane<6, 1, 1>, 2, 1, -1>(),
    traj_inst<FiberLane<4, 2, 1, 0>, 1>(), traj_inst<FiberLane<4, 1, 1, 0>, 1>(), traj_inst<FiberLane<4, 1, 1, 0>, 2>(), traj_inst<FiberLane<2, 1, 1, 0>, 1>(),   // general Hanti (AS = 0)
    traj_inst<FiberLane<5, 3, 1>, 1, 1, 0, 0, 0, 8>(), traj_inst<FiberLane<4, 3, 1>, 1, 1, 0, 0, 0, 8>(), traj_inst<FiberLane<3, 3, 1>, 1, 1, 0, 0, 0, 8>(),   // trajectories of 5 ... 8 warps (e.g. 45 x 12)
};
const InstPart kInstC = inst_part(kInst);
