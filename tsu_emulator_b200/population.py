"""
Estimators of population annealing that do not depend on the model: ln Z ratios, free energies and the family
statistic, shared by the lattice (lattice.PopulationResult) and the dense and sparse sampler
(gibbs.DensePopulationResult).
"""

import math

import numpy as np


class PopulationEstimates:
    """Base of the population-annealing results.  A subclass sets (P = n_populations, n = len(temperatures)):
      weight_sum    int64 device tensor [n, P], W = sum of the quantised weights floor(exp(-dbeta (E_i - E_ref)) 2^s)
      energy_ref    float64 device tensor [n, P], E_ref = lowest E of the population entering step k
      family        int32 device tensor [n_chains], the initial member each member descends from
      temperatures  float64 [n], T_start, dbeta float64 [n], r_pop (R_p), shift (s), n_sites (N)
    """

    @property
    def n_populations(self) -> int:
        return int(self.weight_sum.shape[1])

    def log_q(self) -> np.ndarray:
        """[n, P] float64: ln Q_k = ln Z(T_k) / Z(T_{k-1}) ~ ln(W / (R_p 2^s)) - dbeta_k E_ref"""
        W = self.weight_sum.cpu().numpy().astype(np.float64)
        e_ref = self.energy_ref.cpu().numpy()
        return np.log(W) - math.log(self.r_pop) - self.shift * math.log(2.0) - self.dbeta[:, None] * e_ref

    def log_z_ratio(self) -> np.ndarray:
        """[n, P]: ln Z(T_k) / Z(T_start), the cumulative sum of log_q"""
        return np.cumsum(self.log_q(), axis=0)

    def free_energy(self) -> np.ndarray:
        """[n, P]: free energy per site -T_k ln Z(T_k) / N, with ln Z(T_start = inf) = N ln 2"""
        if not math.isinf(self.T_start):
            raise ValueError("free_energy needs a run from T_start = inf (ln Z is known only at infinite temperature)")
        N = self.n_sites
        return -self.temperatures[:, None] * (N * math.log(2.0) + self.log_z_ratio()) / N

    def rho_t(self) -> np.ndarray:
        """[P]: R_p sum_f (n_f / R_p)^2 over the families f of each population (1 when every family has one member)"""
        fam = self.family.cpu().numpy().reshape(self.n_populations, self.r_pop)
        out = np.empty(self.n_populations)
        for p in range(self.n_populations):
            n_f = np.unique(fam[p], return_counts=True)[1].astype(np.float64)
            out[p] = (n_f * n_f).sum() / self.r_pop
        return out
