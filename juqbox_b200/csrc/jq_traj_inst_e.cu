// Part of the instantiation table of the register-resident trajectory kernels (see jq_traj_kernels.cuh): segment sweeps of the
// time-parallel evaluation (jq_seg.cu), tile layouts.
#include "jq_traj_kernels.cuh"

template <int NC, int NT, int JT = 0, int GLT = 0, int NW = TRAJ_WARPS>
constexpr Inst tile_seg() { return traj_inst<TileLane<NC, NT>, 1, 1, JT, 0, GLT, NW, 0, true>(); }

const Inst kInst[] = {
    tile_seg<2, 0, 4, 32>(), tile_seg<2, 0>(),       // 4 x 4 levels, one element per lane (cnot2 example shape: J = 4)
    tile_seg<3, 1, 3, 32>(), tile_seg<3, 1>(),       // 4 x 4 x 4 levels, two elements per lane (cnot3 example shape: J = 3)
    tile_seg<2, 2, 4, 16>(), tile_seg<2, 2>(),       // throughput layouts for the propagator launch (many unit-vector sweeps)
    tile_seg<3, 3, 3, 32, 8>(), tile_seg<3, 3, 0, 0, 8>(),
};
const InstPart kInstE = inst_part(kInst);
