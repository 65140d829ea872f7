"""One resampling step of population annealing on any chain states (tsu_population_resample), restated for the tests
from the pieces of the lattice oracle (oracle/population_oracle.py): quantised_weight, systematic_parents and
resample_draw.  Imported by the dense population tests; not a test module itself."""
import numpy as np

from oracle import population_oracle as PO


def resample_populations(energy, family, dbeta, seed, chain0, sweep, P):
    """steps 2-4 of one step on n chains in P equal contiguous populations: energy [n] float64, family [n] ints, dbeta
    float64, the draw of population p at (sweep, chain0 + p R_p), wrapping mod 2^32.  Returns (parents [n], the global
    index each child copies; family [n] of the children; W [P] Python ints; E_ref [P])."""
    energy = np.asarray(energy, dtype=np.float64)
    n = len(energy)
    r_pop = n // int(P)
    s = PO.weight_shift(r_pop)
    parents = np.empty(n, dtype=np.int64)
    W, e_ref = [], np.empty(int(P))
    for p in range(int(P)):
        lo = p * r_pop
        E = energy[lo:lo + r_pop]
        e_ref[p] = min(E)
        q = [PO.quantised_weight(float(dbeta) * (float(e) - e_ref[p]), s) for e in E]
        par, w = PO.systematic_parents(q, PO.resample_draw(seed, chain0 + lo, sweep))
        parents[lo:lo + r_pop] = lo + np.asarray(par, dtype=np.int64)
        W.append(w)
    return parents, [int(family[i]) for i in parents], W, e_ref
