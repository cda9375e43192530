"""Oracle-backed stand-in for the CUDA trajectory store in data-augmented MCMC (dpomp_b200.MbpParticles.da_loglike / da_step),
used to test the host-side run_std_mcmc driver on CPU and as the checker of the GPU chains.  Same duck-typed interface as the
device store; trajectories live in numpy, the walks and proposals are those of oracle/dpomp_oracle_da.c."""
import numpy as np

from fake_mbp import OracleMbp
from oracle import da_oracle as dao


class OracleDa(OracleMbp):
    def __init__(self, desc, obs_times, t0_index, n, cap=4096, seed=1, max_traj=196000):
        super().__init__(desc, obs_times, t0_index, n, cap, seed)
        self.max_traj = int(max_traj)

    def iterate(self, theta, obs_i, fresh):
        theta = np.asarray(theta, dtype=np.float64)
        out = np.zeros(theta.shape[1])
        for p in range(theta.shape[1]):
            if fresh:
                self.fc[p] = self.ic; self.len[p] = 0; self.ll[p] = 0.0
            t_start = (theta[self.t0_index - 1, p] if self.t0_index > 0 else 0.0) if obs_i == 1 else self.obs_times[obs_i - 2]
            out[p], self.len[p] = dao.mbp_iterate(self.desc, theta[:, p], self.fc[p], self.t[p], self.y[p], self.len[p], self.ll[p],
                                                  t_start, obs_i, self.key, self.offset + p)
        return out

    def da_loglike(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        return np.array([dao.da_loglike(self.desc, theta[:, p], self.t[p, : self.len[p]], self.y[p, : self.len[p]])[0]
                         for p in range(theta.shape[1])])

    def da_step(self, theta_cur, theta_f, kind, traj_props, mvp):
        theta_cur = np.asarray(theta_cur, dtype=np.float64); theta_f = np.asarray(theta_f, dtype=np.float64)
        n = theta_cur.shape[1]
        out = np.full((n, 2), -np.inf)
        acc = np.zeros((n, 3), dtype=np.int64)
        for p in range(n):
            if kind[p] == 0:
                out[p] = dao.da_loglike(self.desc, theta_f[:, p], self.t[p, : self.len[p]], self.y[p, : self.len[p]])[0]
            elif kind[p] == 1:
                assert self.len[p] + traj_props <= self.cap, "OracleDa: raise cap"
                self.len[p], self.fc[p], self.ll[p], acc[p] = dao.da_props(self.desc, theta_cur[:, p], self.t[p], self.y[p], self.len[p],
                                                                           self.max_traj, traj_props, mvp, self.key, self.offset + p)
                out[p] = self.ll[p]
        return out, acc
