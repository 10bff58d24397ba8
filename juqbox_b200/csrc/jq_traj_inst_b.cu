// Part of the instantiation table of the register-resident trajectory kernels (see jq_traj_kernels.cuh).
#include "jq_traj_kernels.cuh"

const Inst kInst[] = {
    traj_inst<SlotLane<1, 2, 1, 2>, 1>(), traj_inst<SlotLane<1, 3, 1, 2>, 1>(), traj_inst<SlotLane<1, 4, 1, 2>, 1>(), traj_inst<SlotLane<1, 4, 2, 2>, 1>(),
    traj_inst<SlotLane<1, 2, 2, 2>, 1>(), traj_inst<SlotLane<2, 2, 3, 2>, 1>(), traj_inst<SlotLane<3, 1, 3, 2>, 1>(), traj_inst<SlotLane<1, 1, 1, 2>, 1>(),
    traj_inst<SlotLane<1, 1, 2, 2>, 1>(),
    traj_inst<SlotLane<1, 4, 2, 2>, 1, 1, 0, 1>(), traj_inst<SlotLane<1, 3, 1, 2>, 1, 1, 0, 1>(),      // objFuncType 2/3
    traj_inst<SlotLane<1, 4, 1, 2>, 1, 1, 0, 1>(), traj_inst<SlotLane<1, 2, 1, 2>, 1, 1, 0, 1>(),
    traj_inst<FiberLane<4, 2, 1, 1, 1>, 1, 1, 4, 0, 16>(),     // cnot2 example shape: warp-shuffle exchange measured 3.5% faster than shared memory
    traj_inst<FiberLane<6, 1, 1>, 2, 1, 3, 0, 4>(),
    traj_inst<FiberLane<4, 3, 1>, 1, 1, 3, 0, 32>(),           // cnot3 example shape (J = 3, 32-lane groups): +2% over the runtime-J kernel; the shuffle twin was 1% slower
    traj_inst<FiberLane<4, 1, 1>, 2, 3, 5, 0, 3>(),            // risk-neutral SWAP 0-2 shape (n = 4, m = 3, J = 5)
};
const InstPart kInstB = inst_part(kInst);
