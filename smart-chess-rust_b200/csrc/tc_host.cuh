// Host-side tensor-map helpers shared by tower_bf16.cu and tower_lat.cu (defined in tower_bf16.cu).
#pragma once
#include <cuda.h>

namespace scb {

// tiled tensor map of 16-bit elements (dt: bf16 or fp16, the kernel's operand type) with 128-byte swizzle; returns
// SC_OK or SC_E_CUDA (message in sc_last_error)
int tc_encode_map(CUtensorMap *m, CUtensorMapDataType dt, const void *ptr, int rank, const cuuint64_t *dims,
                  const cuuint64_t *strides, const cuuint32_t *box, const char *what, bool swizzle128 = true);
// 16-bit NHWC activations [boards][8 ranks][8 files][c] viewed as {C, file, board, rank}: a box of 64 channels x 8 files x
// 2 boards x 10 ranks lands in shared memory with rows ordered (rank, board, file), so the three dy taps of a 3x3
// convolution are 2 KB apart in ONE box (ranks -1 and 8 are zero-filled = the padding)
int tc_make_act_map_hbw(CUtensorMapDataType dt, const void *ptr, int boards, int c, CUtensorMap *m);

}  // namespace scb
