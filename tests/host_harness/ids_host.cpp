// ids_host.cpp -- CPU harness for action ids (doudizhu-rl_b200/csrc/ddz_ids.cuh).
// TEST INFRASTRUCTURE ONLY: compiles the product's id code (block table, ranking, round trip, unranking) for the host with
// g++ (-DDDZ_HOST_HARNESS), so that tests/ can compare it with the oracle's universe where there is no GPU.  Nothing in the
// product loads this.
#define DDZ_HOST_HARNESS
#include <cstdint>
#include <cstring>
#include "../../doudizhu-rl_b200/csrc/ddz_ids.cuh"

using namespace ddz;

extern "C" void ids_host_move_ids(const uint64_t* moves, long long n, int32_t* ids) {
    for (long long i = 0; i < n; i++) ids[i] = move_id(moves[i]);
}
extern "C" void ids_host_moves_of_ids(const int32_t* ids, long long n, uint64_t* moves) {
    for (long long i = 0; i < n; i++) moves[i] = move_of_id(ids[i]);
}
extern "C" int ids_host_blocks(uint64_t* out) {
    memcpy(out, kIdBlocks, sizeof kIdBlocks);
    return DDZ_ID_BLOCKS;
}
