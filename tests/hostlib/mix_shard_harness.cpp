// Host build of the sharded-mix helpers (csrc/mix.cuh): the range -> per-member counts split and the window-geometry bound
// (tests only; never shipped).
#include "mix.cuh"
using namespace h2v;
extern "C" {
int x_shard_counts(u32 members, const u32* global_counts, unsigned long long base, u32 n, u32* local) {
  return mix_shard_counts(members, global_counts, base, n, local) ? 1 : 0;
}
// out[0] = right-channel bound, out[1] = left-channel bound
void x_shard_bound(u32 members, const u32* P, const u32* n_mo, const u32* Sh, const u32* global_counts, u32 max_shard, unsigned long long* out) {
  mix_shard_bound(members, P, n_mo, Sh, global_counts, max_shard, out, out + 1);
}
}
