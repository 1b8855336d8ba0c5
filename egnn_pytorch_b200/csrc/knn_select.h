// Neighbour-select stage of a layer with k > 0 (knn_select.cu).
#pragma once
#include "common.cuh"

namespace egnn {

// Neighbour lists of every row (egnn_pytorch.py:237-260).  In edge-list mode (io.nbr_idx set) `idx` becomes the caller's
// lists and `ok` nullptr; otherwise the lists are ranked into `idx` / `ok`, on coordinates of type `coors_dtype`.
int select_neighbours(const EgnnLayerDesc& d, const Dims& s, const EgnnLayerIO& io, int32_t coors_dtype, int32_t*& idx,
                      uint8_t*& ok, cudaStream_t st);

}  // namespace egnn
