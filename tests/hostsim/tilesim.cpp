// tilesim.cpp - TEST HARNESS ONLY (never shipped, never used by tactics2d_b200).
//
// Compiles the map tile compiler of tactics2d_b200/csrc/t2d_tile.h with g++ so that the blobs K1 and the lidar kernel
// read can be checked on a machine without a GPU (`pytest -m "not gpu"`).  The CUDA library includes the same header.
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "../../tactics2d_b200/csrc/t2d_tile.h"

using namespace t2d;

extern "C" {

// offsets == NULL: compile_tile(tiles[0]); else compile_map_table, and offsets [n_tiles] receives the tiles' byte offsets.
// The result goes to out[cap]; *n_out receives its length (copied only when it fits), err[err_cap] the error text.
int ts_compile(const t2d_map_tile* tiles, int n_tiles, float cell_size, float reach, unsigned char* out, int64_t cap,
               int64_t* n_out, uint32_t* offsets, char* err, int err_cap) {
  std::vector<unsigned char> blob;
  std::vector<uint32_t> offs;
  std::string msg;
  const int r = !offsets ? compile_tile(tiles[0], cell_size, reach, blob, msg)
                         : compile_map_table(tiles, n_tiles, cell_size, reach, blob, offs, msg);
  snprintf(err, (size_t)err_cap, "%s", msg.c_str());
  *n_out = (int64_t)blob.size();
  if (r == T2D_OK && (int64_t)blob.size() <= cap) memcpy(out, blob.data(), blob.size());
  if (r == T2D_OK && offsets) memcpy(offsets, offs.data(), offs.size() * sizeof(uint32_t));
  return r;
}

}
