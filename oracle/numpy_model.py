"""Second, independent restatement of the reference's fit-and-evaluate path -- TEST INFRASTRUCTURE ONLY.

Written directly from /root/reference/src/splpak.F90 (NOT from oracle/splpak_oracle.c) so that the C oracle and
this model can only agree through the Fortran text they both follow: tests/test_oracle_double.py runs both on
random 1-D..4-D problems and asserts bit-equal least-squares rows, coefficients equal to a few ulp*cond, and
equal splde values for every derivative order.  Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may
import this module; the product (splpak_b200/) never does.

Arithmetic: Python floats are IEEE binary64 and CPython never contracts a*b+c into an FMA, so `bascmp`,
the index boxes and the row values below are bit-identical to an unfused real64 Fortran build.  `suprls` uses
numpy slices for its strided inner loops (same algorithm and pivot/sign choices, summation order may differ).

  bascmp   src/splpak.F90:206-389      splcw  :709-1058 (data rows :788-855, histogram :885-907 incl. the bare
  suprls   :1425-1693                         `cycle` of :899, constraint rows :921-1046, final solve :1051-1058)
  splde    :1166-1238                  splfe  :1272-1273           splcc  :440-444
"""
from __future__ import annotations

import math

import numpy as np


def _trunc(v: float) -> int:
    """Fortran real -> default-integer assignment / int(): truncation toward zero."""
    return int(v)


class SplpakModel:
    """State that the reference keeps in splpak_type (:95-111)."""

    def __init__(self):
        self.mdim = 0
        self.dx = []
        self.dxin = []
        self.ib = []
        self.ibmn = []
        self.ibmx = []
        # suprls cursor
        self.ilast = self.isav = self.iold = self.np1 = self.l = self.il1 = self.k = self.k1 = 0
        self.errsum = 0.0

    # ------------------------------------------------------------------ bascmp :206-389
    def bascmp(self, x, nderiv, xmin, nodes):
        icol = 0
        basm = 1.0
        m = self.mdim
        for idim in range(1, m + 1):
            mdmid = m + 1 - idim
            icol = nodes[mdmid - 1] * icol + self.ib[mdmid - 1]                 # :227
            ibd = self.ib[idim - 1]
            ntyp = 1
            if ibd > 1:
                ntyp = 2
                if ibd >= nodes[idim - 1] - 2:
                    ntyp = 3
            ngo = 3 * ntyp + nderiv[idim - 1] - 2                               # :243
            dxin = self.dxin[idim - 1]
            xd = x[idim - 1]
            xb = xmin[idim - 1] + float(ibd) * self.dx[idim - 1]                # :246
            bas1 = 0.0
            if ngo == 4:                                                        # :253-270
                z = abs(dxin * (xd - xb)) - 2.0
                if z < 0.0:
                    bas1 = -0.25 * (z * z * z)
                    z = z + 1.0
                    if z < 0.0:
                        bas1 = bas1 + z * z * z
            elif ngo == 5:                                                      # :272-286
                z = xd - xb
                fact = dxin
                if z < 0.0:
                    fact = -fact
                z = fact * z - 2.0
                if z < 0.0:
                    bas1 = -0.75 * (z * z)
                    z = z + 1.0
                    if z < 0.0:
                        bas1 = bas1 + 3.0 * (z * z)
                    bas1 = fact * bas1
            elif ngo == 6:                                                      # :288-300
                fact = dxin
                z = fact * abs(xd - xb) - 2.0
                if z < 0.0:
                    bas1 = -1.5 * z
                    z = z + 1.0
                    if z < 0.0:
                        bas1 = bas1 + 6.0 * z
                    bas1 = (fact * fact) * bas1
            elif ngo in (2, 8):                                                 # :302-322
                fact = -dxin if ngo == 2 else dxin
                z = fact * (xd - xb) + 2.0
                if z > 0.0:
                    if z < 2.0:
                        bas1 = 1.5 * (z * z)
                        z = z - 1.0
                        if z > 0.0:
                            bas1 = bas1 - 3.0 * (z * z)
                        bas1 = fact * bas1
                    else:
                        bas1 = 3.0 * fact
            elif ngo in (3, 9):                                                 # :324-340
                fact = -dxin if ngo == 3 else dxin
                z = fact * (xd - xb) + 2.0
                z1 = z - 1.0
                if abs(z1) < 1.0:
                    bas1 = 3.0 * z
                    if z1 > 0.0:
                        bas1 = bas1 - 6.0 * z1
                    bas1 = (fact * fact) * bas1
            else:                                                               # case default :342-379
                if ngo != 7:
                    z = dxin * (xb - xd) + 2.0
                else:
                    z = dxin * (xd - xb) + 2.0
                if z > 0.0:
                    if z < 2.0:
                        bas1 = 0.5 * (z * z * z)
                        z = z - 1.0
                        if z > 0.0:
                            bas1 = bas1 - z * z * z
                    else:
                        bas1 = 3.0 * z - 3.0
            basm = basm * bas1                                                  # :383
        return icol + 1, basm                                                   # :387

    def _odometer(self):
        """Advance me%ib inside [ibmn, ibmx], dimension 1 fastest; False when the box is exhausted (:840-846)."""
        for idim in range(self.mdim):
            self.ib[idim] += 1
            if self.ib[idim] <= self.ibmx[idim]:
                return True
            self.ib[idim] = self.ibmn[idim]
        return False

    # ------------------------------------------------------------------ row generation of splcw
    def _setup(self, ndim, xmin, xmax, nodes):
        self.mdim = ndim
        self.dx = [0.0] * ndim
        self.dxin = [0.0] * ndim
        self.ib = [0] * ndim
        self.ibmn = [0] * ndim
        self.ibmx = [0] * ndim
        ncol = 1
        for idim in range(ndim):
            nod = nodes[idim]
            ncol *= nod
            xrng = xmax[idim] - xmin[idim]
            self.dx[idim] = xrng / float(nod - 1)                               # :747
            self.dxin[idim] = 1.0 / self.dx[idim]                               # :748
        return ncol

    def rows(self, ndim, xdata, ydata, wdata, xmin, xmax, nodes, xtrap):
        """Every least-squares row the reference hands to suprls, in order: list of (dict col0->value, rhs).
        xdata[i] is point i; wdata None or wdata[0] < 0 means unweighted (:796)."""
        nodes = [int(v) for v in nodes]
        xmin = [float(v) for v in xmin]
        xmax = [float(v) for v in xmax]
        ncol = self._setup(ndim, xmin, xmax, nodes)
        ndata = len(ydata)
        weighted = wdata is not None and len(wdata) > 0 and float(wdata[0]) >= 0.0
        out = []
        nderiv = [0] * ndim
        for idata in range(ndata):                                              # :788-855
            rowwt = 1.0
            if weighted:
                rowwt = float(wdata[idata])
                if rowwt == 0.0:
                    continue
            rhs = rowwt * float(ydata[idata])
            x = [float(xdata[idata][d]) for d in range(ndim)]
            for idim in range(ndim):
                nod = nodes[idim]
                it = _trunc(self.dxin[idim] * (x[idim] - xmin[idim]))           # :822
                self.ibmn[idim] = min(max(it - 1, 0), nod - 2)
                self.ib[idim] = self.ibmn[idim]
                self.ibmx[idim] = max(min(it + 2, nod - 1), 1)
            row = {}
            while True:
                icol, basm = self.bascmp(x, nderiv, xmin, nodes)
                row[icol - 1] = rowwt * basm                                    # :837
                if not self._odometer():
                    break
            out.append((row, rhs))
        if xtrap != 0.0:                                                        # :862-1048
            inmx = [nodes[d] - 1 for d in range(ndim)]
            nrect = 1
            for d in range(ndim):
                nrect *= inmx[d]
            work, totlwt = self.histogram(ndim, xdata, wdata, xmin, xmax, nodes)
            wtprrc = totlwt / float(nrect)                                      # :910
            inn = [0] * ndim
            iin = 0
            spcrit = 0.75
            while True:                                                         # node_index :921-1046
                iin += 1
                expect = wtprrc
                for d in range(ndim):
                    if inn[d] == 0 or inn[d] == inmx[d]:
                        expect = 0.5 * expect
                if work[iin - 1] < spcrit * expect:
                    dcwght = expect - work[iin - 1]
                    x = [0.0] * ndim
                    for d in range(ndim):
                        ini = inn[d]
                        x[d] = xmin[d] + float(ini) * self.dx[d]
                        self.ibmn[d] = ini - 1
                        self.ibmx[d] = ini + 1
                        if ini == 0:
                            self.ibmn[d] = 0
                        if ini == inmx[d]:
                            self.ibmx[d] = inmx[d]
                        self.ib[d] = self.ibmn[d]
                    dcwght = xtrap * dcwght
                    for idm in range(ndim):
                        for jdm in range(idm, ndim):
                            nderiv = [0] * ndim
                            boundary = True
                            rowwt = 2.0 * dcwght
                            if jdm == idm:
                                rowwt = dcwght
                                nderiv[jdm] = 2
                                if inn[idm] != 0 and inn[idm] != inmx[idm]:
                                    boundary = False
                            if boundary:
                                nderiv[idm] = 1
                                nderiv[jdm] = 1
                            row = {}
                            while True:
                                icol, basm = self.bascmp(x, nderiv, xmin, nodes)
                                row[icol - 1] = rowwt * basm
                                if not self._odometer():
                                    break
                            out.append((row, 0.0))
                    nderiv = [0] * ndim
                # advance the node odometer
                done = True
                for d in range(ndim):
                    inn[d] += 1
                    if inn[d] <= inmx[d]:
                        done = False
                        break
                    inn[d] = 0
                if done:
                    break
        return out, ncol

    def histogram(self, ndim, xdata, wdata, xmin, xmax, nodes):
        """The nearest-node weight histogram of :885-907: (work[ncol], totlwt).  Same weight convention as rows."""
        nodes = [int(v) for v in nodes]
        xmin = [float(v) for v in xmin]
        xmax = [float(v) for v in xmax]
        ncol = self._setup(ndim, xmin, xmax, nodes)
        weighted = wdata is not None and len(wdata) > 0 and float(wdata[0]) >= 0.0
        inmx = [nodes[d] - 1 for d in range(ndim)]
        work = [0.0] * ncol
        totlwt = 0.0
        for idata in range(len(xdata)):                                         # :885-907
            bump = 1.0
            if weighted:
                bump = float(wdata[idata])
            if bump == 0.0:
                continue
            iin = 0
            for idimc in range(1, ndim + 1):
                idim = ndim + 1 - idimc
                inidim = _trunc(self.dxin[idim - 1] * (float(xdata[idata][idim - 1]) - xmin[idim - 1]) + 0.5)
                if inidim < 0 or inidim > inmx[idim - 1]:
                    continue                                                    # the bare `cycle` of :899: this dimension is dropped
                iin = (inmx[idim - 1] + 1) * iin + inidim
            work[iin] = work[iin] + bump
            totlwt = totlwt + bump
        return work, totlwt

    # ------------------------------------------------------------------ suprls :1425-1693 (1-based scratch a[1..nn])
    def suprls(self, i, rowi, n, bi, a, nn, soln):
        """Returns (ier, err).  a is a numpy array of length nn+1 (index 0 unused)."""
        tol = 1.0e-18
        complete = i <= 0
        if not complete:
            if i <= 1:
                self.iold = 0
                self.np1 = n + 1
                self.l = nn // self.np1
                self.ilast = 0
                self.il1 = 0
                self.k = 0
                self.k1 = 0
                self.errsum = 0.0
                nreq = ((n + 5) * n + 2) // 2
                if nn < nreq:
                    return 32, 0.0
            if i - self.iold != 1:
                return 35, 0.0
            self.iold = i
            a[self.ilast + 1:self.ilast + n + 1] = rowi
            a[self.ilast + self.np1] = bi
            self.ilast += self.np1
            self.isav = i
            if i < self.l:
                return 0, 0.0
        np1 = self.np1
        while True:
            if not complete:
                if self.k != 0:
                    self.k1 = min(self.k, n)
                    idiag = -np1
                    if self.l - self.k == 1:                                    # Givens :1488-1515
                        for j in range(1, self.k1 + 1):
                            idiag += np1 - j + 2
                            i1 = self.il1 + j
                            if abs(a[i1]) <= tol:
                                s = math.sqrt(a[idiag] * a[idiag])
                            elif abs(a[idiag]) < tol:
                                s = math.sqrt(a[i1] * a[i1])
                            else:
                                s = math.sqrt(a[idiag] * a[idiag] + a[i1] * a[i1])
                            if s == 0.0:
                                continue
                            temp = a[idiag]
                            a[idiag] = s
                            s = 1.0 / s
                            cn = temp * s
                            sn = a[i1] * s
                            cnt = np1 - j                                       # j1 = j+1 .. np1
                            if cnt > 0:
                                top = a[idiag + 1:idiag + 1 + cnt].copy()
                                bot = a[i1 + 1:i1 + 1 + cnt].copy()
                                a[idiag + 1:idiag + 1 + cnt] = cn * top + sn * bot
                                a[i1 + 1:i1 + 1 + cnt] = -sn * top + cn * bot
                    else:                                                       # Householder :1516-1549
                        nrow = self.l - self.k
                        for j in range(1, self.k1 + 1):
                            idiag += np1 - j + 2
                            i1 = self.il1 + j
                            col = a[i1:i1 + np1 * (nrow - 1) + 1:np1]
                            s = a[idiag] * a[idiag] + float(np.dot(col, col))
                            if s == 0.0:
                                continue
                            temp = a[idiag]
                            a[idiag] = math.sqrt(s)
                            if temp > 0.0:
                                a[idiag] = -a[idiag]
                            temp = temp - a[idiag]
                            temp1 = 1.0 / (temp * a[idiag])
                            cnt = np1 - j
                            if cnt > 0:
                                # rows of the new block restricted to columns j+1..np1: element (r, jdel) at i1 + r*np1 + jdel
                                blk = np.lib.stride_tricks.as_strided(
                                    a[i1 + 1:], shape=(nrow, cnt), strides=(a.strides[0] * np1, a.strides[0]))
                                top = a[idiag + 1:idiag + 1 + cnt]
                                sv = (temp * top + col @ blk) * temp1
                                top += sv * temp
                                blk += np.outer(col, sv)
                    if self.k >= n:                                             # :1551-1566
                        lmkm1 = self.l - self.k
                        for ii in range(1, lmkm1 + 1):
                            ilnp = self.il1 + ii * np1
                            self.errsum += a[ilnp] * a[ilnp]
                        if i <= 0:
                            break
                        self.k = self.l
                        self.ilast = self.il1
                        self.l = self.k + (nn - self.ilast) // np1
                        return 0, 0.0
                k11 = self.k1 + 1
                self.k1 = min(self.l, n)
                if self.l - self.k != 1:                                        # :1569-1619
                    k1m1 = self.k1 - 1
                    if self.l > n:
                        k1m1 = n
                    i1 = self.il1 + k11 - np1 - 1
                    for j in range(k11, k1m1 + 1):
                        i1 += np1 + 1
                        i2 = i1 + (self.l - j) * np1
                        col = a[i1:i2 + 1:np1]
                        s = float(np.dot(col, col))
                        if s == 0.0:
                            continue
                        temp = a[i1]
                        a[i1] = math.sqrt(s)
                        if temp > 0.0:
                            a[i1] = -a[i1]
                        temp = temp - a[i1]
                        temp1 = 1.0 / (temp * a[i1])
                        cnt = np1 - j
                        nbelow = (i2 - i1) // np1
                        if cnt > 0:
                            top = a[i1 + 1:i1 + 1 + cnt]
                            if nbelow > 0:
                                below = a[i1 + np1:i2 + 1:np1]
                                blk = np.lib.stride_tricks.as_strided(
                                    a[i1 + np1 + 1:], shape=(nbelow, cnt), strides=(a.strides[0] * np1, a.strides[0]))
                                sv = (temp * top + below @ blk) * temp1
                                top += sv * temp
                                blk += np.outer(below, sv)
                            else:
                                sv = (temp * top) * temp1
                                top += sv * temp
                    if self.l > n:
                        np1mk = np1 - self.k
                        lmk = self.l - self.k
                        for ii in range(np1mk, lmk + 1):
                            ilnp = self.il1 + ii * np1
                            self.errsum += a[ilnp] * a[ilnp]
                imov = 0                                                        # squeeze :1620-1635
                i1 = self.il1 + k11 - np1 - 1
                i2 = i1
                for ii in range(k11, self.k1 + 1):
                    imov += ii - 1
                    i1 += np1 + 1
                    i2 = i1 + np1 - ii
                    a[i1 - imov:i2 - imov + 1] = a[i1:i2 + 1].copy()
                self.ilast = i2 - imov
                self.il1 = self.ilast
                if i <= 0:
                    break
                self.k = self.l
                self.l = self.k + (nn - self.ilast) // np1
                return 0, 0.0
            complete = False                                                    # :1645-1659
            self.l = self.isav
            if self.l < n:
                return 33, 0.0
            if self.k == self.isav:
                break
        self.ilast = (np1 * (np1 + 1)) // 2 - 1                                 # back-substitution :1661-1690
        if a[self.ilast - 1] == 0.0:
            return 34, 0.0
        soln[n - 1] = a[self.ilast] / a[self.ilast - 1]
        for ii in range(2, n + 1):
            self.ilast -= ii
            s = a[self.ilast]
            for k in range(1, ii):
                s = s - a[self.ilast - k] * soln[np1 - k - 1]
            ilii = self.ilast - ii
            if a[ilii] == 0.0:
                return 34, 0.0
            soln[np1 - ii - 1] = s / a[ilii]
        return 0, math.sqrt(self.errsum)

    # ------------------------------------------------------------------ splcw / splcc
    def splcw(self, ndim, xdata, ydata, wdata, xmin, xmax, nodes, xtrap, nwrk=None):
        """Returns (coef, ierror).  Validation order :718-781."""
        if ndim < 1:
            return None, 101
        ncol = 1
        for d in range(ndim):
            if nodes[d] < 4:
                return None, 102
            ncol *= int(nodes[d])
            if float(xmax[d]) - float(xmin[d]) == 0.0:
                return None, 103
        if len(ydata) < 1:
            return None, 105
        if nwrk is None:
            nwrk = ncol * (ncol + 1) + 1
        nwrk1 = ncol + 1 if xtrap != 0.0 else 1
        nwlft = nwrk - nwrk1 + 1
        if nwlft < 1:
            return None, 106
        rows, ncol = self.rows(ndim, xdata, ydata, wdata, xmin, xmax, nodes, xtrap)
        a = np.zeros(nwlft + 1)
        coef = np.zeros(ncol)
        ierror = 0
        irow = 0
        dense = np.zeros(ncol)
        for row, rhs in rows:
            irow += 1
            dense[:] = 0.0
            for c, v in row.items():
                dense[c] = v
            ier, _ = self.suprls(irow, dense, ncol, rhs, a, nwlft, coef)
            if ier != 0:
                ierror = 107
        ier, _ = self.suprls(0, dense, ncol, 0.0, a, nwlft, coef)
        if ier != 0:
            ierror = 107
        return coef, ierror

    def splcc(self, ndim, xdata, ydata, xmin, xmax, nodes, xtrap, nwrk=None):
        return self.splcw(ndim, xdata, ydata, [-1.0], xmin, xmax, nodes, xtrap, nwrk)   # :440-444

    # ------------------------------------------------------------------ splde / splfe :1166-1238, :1272
    def splde(self, ndim, x, nderiv, coef, xmin, xmax, nodes):
        """Returns (value, ierror)."""
        ierror = 0
        if ndim < 1:
            return 0.0, 101
        self.mdim = ndim
        self.dx = [0.0] * ndim
        self.dxin = [0.0] * ndim
        self.ib = [0] * ndim
        self.ibmn = [0] * ndim
        self.ibmx = [0] * ndim
        iibmx = 1
        for d in range(ndim):
            nod = int(nodes[d])
            if nod < 4:
                return 0.0, 102
            xrng = float(xmax[d]) - float(xmin[d])
            if xrng == 0.0:
                return 0.0, 103
            if nderiv[d] < 0 or nderiv[d] > 2:
                ierror = 104                                                    # no return (:1190-1194)
            self.dx[d] = xrng / float(nod - 1)
            self.dxin[d] = 1.0 / self.dx[d]
            it = _trunc(self.dxin[d] * (float(x[d]) - float(xmin[d])))
            self.ibmn[d] = min(max(it - 1, 0), nod - 2)
            self.ibmx[d] = max(min(it + 2, nod - 1), 1)
            iibmx *= self.ibmx[d] - self.ibmn[d] + 1
            self.ib[d] = self.ibmn[d]
        total = 0.0
        xs = [float(v) for v in x]
        mn = [float(v) for v in xmin]
        nd = [int(v) for v in nderiv]
        no = [int(v) for v in nodes]
        iib = 0
        while True:
            iib += 1
            icof, basm = self.bascmp(xs, nd, mn, no)
            total = total + float(coef[icof - 1]) * basm                        # :1225
            if iib < iibmx and self._odometer():
                continue
            break
        return total, ierror

    def splfe(self, ndim, x, coef, xmin, xmax, nodes):
        return self.splde(ndim, x, [0] * max(ndim, 0), coef, xmin, xmax, nodes)


# ------------------------------------------------------------------------------------------------------------------
# Vectorised numpy form of the SAME basis arithmetic (value only, nderiv = 0) for large samples: used by bench.py's
# "algorithm-matched" CPU baseline (sparse normal equations + banded Cholesky), not by any parity test.
# ------------------------------------------------------------------------------------------------------------------
def window_weights_numpy(x, xmin, xmax, nod):
    """For a vector of coordinates: window start ws (clamp(it-1, 0, nod-4)) and the 4 basis values of nodes
    ws..ws+3, same formulas as bascmp's value cases (:253-270, :342-379)."""
    dx = (xmax - xmin) / float(nod - 1)
    dxin = 1.0 / dx
    it = np.trunc(dxin * (x - xmin)).astype(np.int64)
    ws = np.clip(it - 1, 0, nod - 4)
    b = np.zeros((4, x.size))
    for k in range(4):
        ib = ws + k
        xb = xmin + ib.astype(np.float64) * dx
        u = dxin * (x - xb)
        left = ib <= 1
        edge = left | (ib >= nod - 2)
        # chapeau
        z = np.abs(u) - 2.0
        v = np.where(z < 0.0, -0.25 * (z * z * z), 0.0)
        z1 = z + 1.0
        v = np.where(z1 < 0.0, v + z1 * z1 * z1, v)
        # edge functions
        ze = np.where(left, -u, u) + 2.0
        ve = np.where(ze > 0.0, 0.5 * (ze * ze * ze), 0.0)
        zm = ze - 1.0
        ve = np.where((ze > 0.0) & (zm > 0.0), ve - zm * zm * zm, ve)
        ve = np.where(ze >= 2.0, 3.0 * ze - 3.0, ve)
        b[k] = np.where(edge, ve, v)
    return ws, b
