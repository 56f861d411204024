"""Writer of the reference's output file `pic1dp.out` (PETSc binary viewer layout, big-endian), fed by the on-device
diagnostics, so that the reference's analysis tools (tools/OutputData.py, runinfo.py, visual.py) read GPU runs
unchanged.

Layout restated from /root/reference/src/pic1dp_output.F90:
  header  (:74-92)   int32 [nspecies, nmode, nx, nv, nx_opd, nv_opd, modes...], float64 [lx, v_max]
  record  (:117-187) float64 [t, int E^2 dx, (sum v^2, sum v^2 p, sum v^2 w) per species], then VecView of
                     field_mode_re, field_mode_im, field_electric, field_chargeden -- each
                     int32 VEC_FILE_CLASSID (1211214), int32 n, float64[n]
          (:457-474) per species float64 markr_xv, total_xv, pertb_xv [nv_opd*nx_opd], markr_v, total_v, pertb_v [nv_opd]
as read by tools/OutputData.py:26-82.
"""
from __future__ import annotations

import numpy as np

VEC_FILE_CLASSID = 1211214


class OutputWriter:
    def __init__(self, path, gpu, nv: int = 128, nx_opd: int = 64, nv_opd: int = 64, v_max: float = 8.0):
        """gpu: pic1dp_b200.Pic1dGpu.  nv = input_nv (written to the header only, src/pic1dp_input.F90:131)."""
        self.gpu = gpu
        self.p = gpu.params
        self.nx_opd, self.nv_opd, self.v_max = nx_opd, nv_opd, float(v_max)
        self.f = open(path, "wb")
        p = self.p
        ints = [p.nspecies, len(gpu.modes), p.nx, nv, nx_opd, nv_opd] + list(gpu.modes)   # the handle's kept modes
        np.asarray(ints, dtype=">i4").tofile(self.f)
        np.asarray([p.lx, self.v_max], dtype=">f8").tofile(self.f)

    def _vec(self, a):
        np.asarray([VEC_FILE_CLASSID, a.size], dtype=">i4").tofile(self.f)
        np.asarray(a, dtype=">f8").tofile(self.f)

    def output_all(self, time: float):
        """output_field + output_ptcldist (src/pic1dp_output.F90:100-189, :196-477) from device-side reductions."""
        sc, dists = self.gpu.output_all(self.nx_opd, self.nv_opd, self.v_max)   # one pass over the markers
        np.asarray(np.concatenate([[time], sc]), dtype=">f8").tofile(self.f)
        fld = self.gpu.get_field()
        for k in ("mode_re", "mode_im", "electric", "chargeden"):
            self._vec(fld[k])
        for s in range(self.p.nspecies):
            d = dists[s]
            for k in ("markr_xv", "total_xv", "pertb_xv", "markr_v", "total_v", "pertb_v"):
                np.asarray(d[k], dtype=">f8").tofile(self.f)
        return sc

    def close(self):
        if self.f:
            self.f.close()
            self.f = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
