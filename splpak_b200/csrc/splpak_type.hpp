// splpak_type.hpp -- C++ host-side mirror of the reference's `splpak_module` interface
// (src/splpak.F90:45-127) over the C ABI of include/splpak_b200.h.
//
// Same names, argument order, argument meaning and error behaviour as the Fortran type-bound
// procedures, so tests written against it read like the reference's own tests:
//
//     splpak::splpak_type solver;
//     solver.initialize(ndim, xdata, l1xdat, ydata, wdata, ndata, xmin, xmax, nodes, xtrap,
//                       coef, ncf, work, nwrk, ierror);                    // generic -> splcw
//     solver.initialize(ndim, xdata, l1xdat, ydata, ndata, xmin, ...);     // generic -> splcc
//     f = solver.evaluate(ndim, x, coef, xmin, xmax, nodes, ierror);       // generic -> splfe
//     f = solver.evaluate(ndim, x, nderiv, coef, xmin, xmax, nodes, ierror); // generic -> splde
//     solver.destroy();
//
// Arrays are laid out as Fortran passes them (column-major, contiguous).  Like the reference, nothing
// throws or stops: `ierror` is set and cfaerr's text (' IERR=' I5, then the message; :399-407) goes
// to stdout.  All arithmetic happens in the CUDA library; this header only forwards.
#pragma once

#include <cstdint>
#include <cstdio>

#include "../../include/splpak_b200.h"

namespace splpak {

using wp = splpak_real;   // splpak_wp (:43)

class splpak_type {
public:
    bool quiet = false;   // not in the reference: suppress cfaerr output (used by tests)

    // generic :: initialize => splcc, splcw (:117)
    void initialize(int ndim, const wp *xdata, int l1xdat, const wp *ydata, const wp *wdata, int ndata,
                    const wp *xmin, const wp *xmax, const int *nodes, wp xtrap, wp *coef, int ncf, wp *work,
                    int nwrk, int &ierror) {
        splcw(ndim, xdata, l1xdat, ydata, wdata, ndata, xmin, xmax, nodes, xtrap, coef, ncf, work, nwrk, ierror);
    }
    void initialize(int ndim, const wp *xdata, int l1xdat, const wp *ydata, int ndata, const wp *xmin,
                    const wp *xmax, const int *nodes, wp xtrap, wp *coef, int ncf, wp *work, int nwrk,
                    int &ierror) {
        splcc(ndim, xdata, l1xdat, ydata, ndata, xmin, xmax, nodes, xtrap, coef, ncf, work, nwrk, ierror);
    }
    // generic :: evaluate => splfe, splde (:118)
    wp evaluate(int ndim, const wp *x, const wp *coef, const wp *xmin, const wp *xmax, const int *nodes,
                int &ierror) {
        return splfe(ndim, x, coef, xmin, xmax, nodes, ierror);
    }
    wp evaluate(int ndim, const wp *x, const int *nderiv, const wp *coef, const wp *xmin, const wp *xmax,
                const int *nodes, int &ierror) {
        return splde(ndim, x, nderiv, coef, xmin, xmax, nodes, ierror);
    }
    // destroy_splpak (:136-165): the GPU path keeps no per-object state between calls
    void destroy() { mdim_ = 0; }
    void destroy(int /*ndim*/) { mdim_ = 0; }

    // ---- the four user entries (:120-123) ----
    void splcc(int ndim, const wp *xdata, int l1xdat, const wp *ydata, int ndata, const wp *xmin,
               const wp *xmax, const int *nodes, wp xtrap, wp *coef, int ncf, wp *work, int nwrk, int &ierror) {
        mdim_ = ndim;
        splpak_b200_splcc(ndim, xdata, l1xdat, ydata, ndata, xmin, xmax, nodes, xtrap, coef, ncf, work, nwrk,
                          &ierror);
        cfaerr(ierror, false);
    }
    void splcw(int ndim, const wp *xdata, int l1xdat, const wp *ydata, const wp *wdata, int ndata,
               const wp *xmin, const wp *xmax, const int *nodes, wp xtrap, wp *coef, int ncf, wp *work,
               int nwrk, int &ierror) {
        mdim_ = ndim;
        splpak_b200_splcw(ndim, xdata, l1xdat, ydata, wdata, ndata, xmin, xmax, nodes, xtrap, coef, ncf, work,
                          nwrk, &ierror);
        cfaerr(ierror, false);
    }
    wp splfe(int ndim, const wp *x, const wp *coef, const wp *xmin, const wp *xmax, const int *nodes,
             int &ierror) {
        mdim_ = ndim;
        const wp f = splpak_b200_splfe(ndim, x, coef, xmin, xmax, nodes, &ierror);
        cfaerr(ierror, true);
        return f;
    }
    wp splde(int ndim, const wp *x, const int *nderiv, const wp *coef, const wp *xmin, const wp *xmax,
             const int *nodes, int &ierror) {
        mdim_ = ndim;
        const wp f = splpak_b200_splde(ndim, x, nderiv, coef, xmin, xmax, nodes, &ierror);
        cfaerr(ierror, true);
        return f;
    }
    // batched evaluation (new entry point; the reference evaluates one point per call)
    void evaluate_batch(int ndim, const wp *x, int l1x, std::int64_t nq, const int *nderiv, const wp *coef,
                        const wp *xmin, const wp *xmax, const int *nodes, wp *out, int &ierror) {
        mdim_ = ndim;
        splpak_b200_eval(ndim, x, l1x, nq, nderiv, coef, xmin, xmax, nodes, out, &ierror);
        cfaerr(ierror, true);
    }
    // every partial derivative up to total order `order` (1 or 2) in one pass: out(ncomp, nq), ncomp = ndim + 1 or
    // (ndim + 1)(ndim + 2) / 2 (new entry point; component k == evaluate_batch with the nderiv it names)
    void evaluate_derivs(int ndim, const wp *x, int l1x, std::int64_t nq, int order, const wp *coef, const wp *xmin,
                         const wp *xmax, const int *nodes, wp *out, int &ierror) {
        mdim_ = ndim;
        splpak_b200_eval_derivs(ndim, x, l1x, nq, order, coef, xmin, xmax, nodes, out, &ierror);
        cfaerr(ierror, true);
    }

private:
    int mdim_ = 0;
    // cfaerr (:399-407)
    void cfaerr(int ierr, bool evaluation) const {
        if (ierr == 0 || quiet) return;
        std::printf(" IERR=%5d\n", ierr);
        std::printf("%s\n", splpak_b200_strerror(ierr, evaluation ? 1 : 0));
    }
};

}   // namespace splpak
