// Lock-free union-find on int32 labels, shared by the lattice cluster moves (ising2d.cu) and the Houdayer move on
// sparse couplings (sparse_houdayer.cu).  Labels form a forest in which a site's parent never has a larger index, so
// every tree's root is its cluster's smallest site index, whatever order the unions run in.  L may lie in shared or
// global memory.
#pragma once
#include <stdint.h>

namespace {

// root of x, halving the path on the way (every site then points at its former grandparent).  A label only ever
// points at a smaller site of the same cluster, so a stale read or an overwritten link still leads to the root
// (the pointer jumping of ECL-CC, Jaiganesh & Burtscher 2018).
__device__ __forceinline__ int cluster_find(int32_t* L, int x) {
  volatile int32_t* V = L;
  int y = V[x];
  while (y != x) {
    const int z = V[y];
    if (z != y) V[x] = z;
    x = y;
    y = z;
  }
  return x;
}

// joins the trees of a and b, hanging the larger root under the smaller (Playne & Hawick's lock-free union)
__device__ __forceinline__ void cluster_union(int32_t* L, int a, int b) {
  while (true) {
    a = cluster_find(L, a);
    b = cluster_find(L, b);
    if (a == b) return;
    if (a > b) {
      const int t = a;
      a = b;
      b = t;
    }
    const int old = atomicMin(L + b, a);
    if (old == b) return;
    b = old;  // b was no longer a root: join its parent (b itself now points to min(old, a)) to a
  }
}

}  // namespace
