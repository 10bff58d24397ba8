// Part of the instantiation table of the register-resident trajectory kernels (see jq_traj_kernels.cuh): segment sweeps of the
// time-parallel evaluation (jq_seg.cu), fibre layouts.
#include "jq_traj_kernels.cuh"

template <int R, int NC, int UPL, int JT = 0, int GLT = 0, int OBJ = 0>
constexpr Inst fiber_seg() { return traj_inst<FiberLane<R, NC, 1>, UPL, 1, JT, OBJ, GLT, TRAJ_WARPS, 0, true>(); }

const Inst kInst[] = {
    fiber_seg<4, 1, 2, 5, 3>(), fiber_seg<4, 1, 2>(), fiber_seg<4, 1, 1>(),      // single qudits: risk-neutral SWAP 0-2 (n = 4, J = 5)
    fiber_seg<6, 1, 2, 3, 4>(), fiber_seg<6, 1, 2>(),                            // cnot1 (n = 6)
    fiber_seg<3, 1, 1>(), fiber_seg<3, 1, 2>(), fiber_seg<5, 1, 2>(), fiber_seg<2, 1, 1>(),
    fiber_seg<4, 2, 1>(), fiber_seg<3, 2, 1>(), fiber_seg<4, 3, 1>(), fiber_seg<3, 3, 1>(),      // coupled qudits without a tile layout
    // objFuncType 2/3: the gradient sweep (mode 5) with the second adjoint set; the other modes run on the instantiations above
    fiber_seg<3, 2, 1, 0, 0, 1>(), fiber_seg<4, 2, 1, 0, 0, 1>(), fiber_seg<4, 1, 1, 0, 0, 1>(), fiber_seg<4, 1, 2, 0, 0, 1>(),
    fiber_seg<6, 1, 2, 0, 0, 1>(), fiber_seg<4, 3, 1, 0, 0, 1>(), fiber_seg<2, 1, 1, 0, 0, 1>(),
};
const InstPart kInstF = inst_part(kInst);
