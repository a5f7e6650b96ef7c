!*****************************************************************************************
!>
!  Drop-in `splpak_module` whose fit-and-evaluate hot path runs on an NVIDIA B200 through
!  the C ABI of `include/splpak_b200.h` (libsplpak_b200.so / libsplpak_b200_r32.so).
!
!  Public surface, names, argument order, kinds and error behaviour are those of the
!  reference module (jacobwilliams/splpak, src/splpak.F90:25-129):
!
!    type(splpak_type) :: s
!    call s%initialize(ndim,xdata,l1xdat,ydata,[wdata,]ndata,xmin,xmax,nodes,xtrap,coef,ncf,work,nwrk,ierror)
!    f = s%evaluate(ndim,x,[nderiv,]coef,xmin,xmax,nodes,ierror)
!    call s%destroy()
!
!  plus additions that have no counterpart in the reference: `evaluate_batch`
!  (batched splfe/splde), `evaluate_derivs` (all partial derivatives up to order 1 or 2 in
!  one pass) and the streaming pair `add_points` / `compute` named by the
!  project brief.  The numerical work (bascmp, the splcw row loop, suprls, splde) is
!  replaced; cfaerr (printing) stays on this side so stdout is unchanged.
!
!  NOTE: no Fortran compiler exists in the build image, so this file is maintained by
!  inspection only; it restricts itself to explicit-shape dummies, value scalars and
!  bind(C) interfaces.  The same C entry points are exercised from C++ and Python tests.
!
!  Build:  gfortran -cpp [-DREAL32] -c splpak_module.F90   and link -lsplpak_b200[_r32]

    module splpak_module

    use iso_fortran_env
    use iso_c_binding

    implicit none

    private

#ifdef REAL32
    integer,parameter :: wp = real32   !! Real working precision [4 bytes]
    integer,parameter :: cwp = c_float
#elif REAL128
#error "splpak_b200: REAL128 has no GPU equivalent (reference src/splpak.F90:37-38)"
#else
    integer,parameter :: wp = real64   !! Real working precision [8 bytes] (default, as the reference)
    integer,parameter :: cwp = c_double
#endif

    integer,parameter,public :: splpak_wp = wp   !! Working precision

    type,public :: splpak_type
        private
        integer :: mdim = 0
        type(c_ptr) :: handle = c_null_ptr      !! streaming fit handle (add_points/compute only)
        contains
        private
        generic,public   :: initialize => splcc, splcw   !! compute the spline coefficients
        generic,public   :: evaluate   => splfe, splde   !! evaluate the spline
        procedure,public :: destroy    => destroy_splpak
        procedure,public :: evaluate_batch               !! (new) batched splfe/splde
        procedure,public :: evaluate_derivs              !! (new) every partial derivative up to order 1 or 2, one pass
        procedure,public :: evaluate_grid                !! (new) splfe/splde on a regular output grid
        procedure,public :: create                       !! (new) streaming fit: create
        procedure,public :: add_points                   !! (new) streaming fit: accumulate points
        procedure,public :: compute                      !! (new) streaming fit: constraints + solve
        procedure,public :: refine                       !! (new) streaming fit: one refinement pass over the same points
        procedure,public :: set_solver                   !! (new) streaming fit: 0 = band Cholesky (default), 1 = orthogonal (Householder)
        procedure,public :: set_smoothing                !! (new) streaming fit: roughness penalty lambda (0 = curvature, 1 = thin plate)
        procedure,public :: enable_gcv                   !! (new) streaming fit: collect what the GCV score needs (before add_points)
        procedure,public :: smoothing_score              !! (new) streaming fit: GCV score {V, RSS, edf, N, ywy} of one lambda
        procedure,public :: select_smoothing             !! (new) streaming fit: lambda minimising the GCV score, set on the fit
        procedure,public :: reml_score                   !! (new) streaming fit: REML score {V_R, D_p, log|M|, n, ywy, phi} of one lambda
        procedure,public :: select_smoothing_reml        !! (new) streaming fit: lambda minimising the REML score, set on the fit
        procedure,public :: prepare_variance             !! (new) streaming fit: tables of the posterior variances (before compute)
        procedure,public :: variance                     !! (new) streaming fit: b(x)^T Sigma b(x) at a batch of points
        procedure,private :: splcc
        procedure,private :: splcw
        procedure,private :: splfe
        procedure,private :: splde
    end type splpak_type

    interface
        function c_splcw(ndim,xdata,l1xdat,ydata,wdata,ndata,xmin,xmax,nodes,xtrap,coef,ncf,work,nwrk,ierror) &
                 bind(C,name='splpak_b200_splcw') result(rc)
            import :: c_int, c_int64_t, cwp
            integer(c_int),value :: ndim, l1xdat
            real(cwp),intent(in) :: xdata(*), ydata(*), wdata(*), xmin(*), xmax(*)
            integer(c_int64_t),value :: ndata, ncf, nwrk
            integer(c_int),intent(in) :: nodes(*)
            real(cwp),value :: xtrap
            real(cwp) :: coef(*), work(*)
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_splcw
        function c_splcc(ndim,xdata,l1xdat,ydata,ndata,xmin,xmax,nodes,xtrap,coef,ncf,work,nwrk,ierror) &
                 bind(C,name='splpak_b200_splcc') result(rc)
            import :: c_int, c_int64_t, cwp
            integer(c_int),value :: ndim, l1xdat
            real(cwp),intent(in) :: xdata(*), ydata(*), xmin(*), xmax(*)
            integer(c_int64_t),value :: ndata, ncf, nwrk
            integer(c_int),intent(in) :: nodes(*)
            real(cwp),value :: xtrap
            real(cwp) :: coef(*), work(*)
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_splcc
        function c_splde(ndim,x,nderiv,coef,xmin,xmax,nodes,ierror) bind(C,name='splpak_b200_splde') result(f)
            import :: c_int, cwp
            integer(c_int),value :: ndim
            real(cwp),intent(in) :: x(*), coef(*), xmin(*), xmax(*)
            integer(c_int),intent(in) :: nderiv(*), nodes(*)
            integer(c_int),intent(out) :: ierror
            real(cwp) :: f
        end function c_splde
        function c_splfe(ndim,x,coef,xmin,xmax,nodes,ierror) bind(C,name='splpak_b200_splfe') result(f)
            import :: c_int, cwp
            integer(c_int),value :: ndim
            real(cwp),intent(in) :: x(*), coef(*), xmin(*), xmax(*)
            integer(c_int),intent(in) :: nodes(*)
            integer(c_int),intent(out) :: ierror
            real(cwp) :: f
        end function c_splfe
        function c_eval(ndim,x,l1x,nq,nderiv,coef,xmin,xmax,nodes,out,ierror) bind(C,name='splpak_b200_eval') result(rc)
            import :: c_int, c_int64_t, c_ptr, cwp
            integer(c_int),value :: ndim, l1x
            integer(c_int64_t),value :: nq
            real(cwp),intent(in) :: x(*), coef(*), xmin(*), xmax(*)
            type(c_ptr),value :: nderiv                      !! c_null_ptr => splfe
            integer(c_int),intent(in) :: nodes(*)
            real(cwp) :: out(*)
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_eval
        function c_eval_derivs(ndim,x,l1x,nq,order,coef,xmin,xmax,nodes,out,ierror) &
                 bind(C,name='splpak_b200_eval_derivs') result(rc)
            import :: c_int, c_int64_t, cwp
            integer(c_int),value :: ndim, l1x, order
            integer(c_int64_t),value :: nq
            real(cwp),intent(in) :: x(*), coef(*), xmin(*), xmax(*)
            integer(c_int),intent(in) :: nodes(*)
            real(cwp) :: out(*)
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_eval_derivs
        function c_eval_grid(ndim,axes,naxis,nderiv,coef,xmin,xmax,nodes,out,ierror) &
                 bind(C,name='splpak_b200_eval_grid') result(rc)
            import :: c_int, c_int64_t, c_ptr, cwp
            integer(c_int),value :: ndim
            real(cwp),intent(in) :: axes(*), coef(*), xmin(*), xmax(*)
            integer(c_int64_t),intent(in) :: naxis(*)
            type(c_ptr),value :: nderiv                      !! c_null_ptr => values (splfe)
            integer(c_int),intent(in) :: nodes(*)
            real(cwp) :: out(*)
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_eval_grid
        function c_fit_create(ndim,xmin,xmax,nodes,xtrap,handle,ierror) bind(C,name='splpak_b200_fit_create') result(rc)
            import :: c_int, c_ptr, cwp
            integer(c_int),value :: ndim
            real(cwp),intent(in) :: xmin(*), xmax(*)
            integer(c_int),intent(in) :: nodes(*)
            real(cwp),value :: xtrap
            type(c_ptr),intent(out) :: handle
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_fit_create
        function c_fit_add_points(h,x,l1x,y,w,weighted,n) bind(C,name='splpak_b200_fit_add_points') result(rc)
            import :: c_int, c_int64_t, c_ptr, cwp
            type(c_ptr),value :: h
            real(cwp),intent(in) :: x(*), y(*), w(*)
            integer(c_int),value :: l1x, weighted
            integer(c_int64_t),value :: n
            integer(c_int) :: rc
        end function c_fit_add_points
        function c_fit_compute(h,coef,ncf,nwrk,ierror) bind(C,name='splpak_b200_fit_compute') result(rc)
            import :: c_int, c_int64_t, c_ptr, cwp
            type(c_ptr),value :: h
            real(cwp) :: coef(*)
            integer(c_int64_t),value :: ncf, nwrk
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_fit_compute
        function c_fit_refine_begin(h) bind(C,name='splpak_b200_fit_refine_begin') result(rc)
            import :: c_int, c_ptr
            type(c_ptr),value :: h
            integer(c_int) :: rc
        end function c_fit_refine_begin
        function c_fit_refine_add_points(h,x,l1x,y,w,weighted,n) bind(C,name='splpak_b200_fit_refine_add_points') result(rc)
            import :: c_int, c_int64_t, c_ptr, cwp
            type(c_ptr),value :: h
            real(cwp),intent(in) :: x(*), y(*), w(*)
            integer(c_int),value :: l1x, weighted
            integer(c_int64_t),value :: n
            integer(c_int) :: rc
        end function c_fit_refine_add_points
        function c_fit_refine_compute(h,coef,ncf,ierror) bind(C,name='splpak_b200_fit_refine_compute') result(rc)
            import :: c_int, c_int64_t, c_ptr, cwp
            type(c_ptr),value :: h
            real(cwp) :: coef(*)
            integer(c_int64_t),value :: ncf
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_fit_refine_compute
        function c_fit_set_solver(h,solver) bind(C,name='splpak_b200_fit_set_solver') result(rc)
            import :: c_int, c_ptr
            type(c_ptr),value :: h
            integer(c_int),value :: solver
            integer(c_int) :: rc
        end function c_fit_set_solver
        function c_fit_set_smoothing(h,lambda,penalty) bind(C,name='splpak_b200_fit_set_smoothing') result(rc)
            import :: c_int, c_double, c_ptr
            type(c_ptr),value :: h
            real(c_double),value :: lambda
            integer(c_int),value :: penalty
            integer(c_int) :: rc
        end function c_fit_set_smoothing
        function c_fit_enable_gcv(h) bind(C,name='splpak_b200_fit_enable_gcv') result(rc)
            import :: c_int, c_ptr
            type(c_ptr),value :: h
            integer(c_int) :: rc
        end function c_fit_enable_gcv
        function c_fit_smoothing_score(h,lambda,penalty,out,nout,ierror) &
                 bind(C,name='splpak_b200_fit_smoothing_score') result(rc)
            import :: c_int, c_double, c_ptr
            type(c_ptr),value :: h
            real(c_double),value :: lambda
            integer(c_int),value :: penalty, nout
            real(c_double),intent(out) :: out(*)
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_fit_smoothing_score
        function c_fit_select_smoothing(h,penalty,lambda_lo,lambda_hi,lambda,out,nout,trace,trace_cap,ntrace,ierror) &
                 bind(C,name='splpak_b200_fit_select_smoothing') result(rc)
            import :: c_int, c_int64_t, c_double, c_ptr
            type(c_ptr),value :: h
            integer(c_int),value :: penalty, nout
            real(c_double),value :: lambda_lo, lambda_hi
            real(c_double),intent(out) :: lambda, out(*), trace(*)
            integer(c_int64_t),value :: trace_cap
            integer(c_int64_t),intent(out) :: ntrace
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_fit_select_smoothing
        function c_fit_reml_score(h,lambda,penalty,out,nout,ierror) &
                 bind(C,name='splpak_b200_fit_reml_score') result(rc)
            import :: c_int, c_double, c_ptr
            type(c_ptr),value :: h
            real(c_double),value :: lambda
            integer(c_int),value :: penalty, nout
            real(c_double),intent(out) :: out(*)
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_fit_reml_score
        function c_fit_select_smoothing_reml(h,penalty,lambda_lo,lambda_hi,lambda,out,nout,trace,trace_cap,ntrace,ierror) &
                 bind(C,name='splpak_b200_fit_select_smoothing_reml') result(rc)
            import :: c_int, c_int64_t, c_double, c_ptr
            type(c_ptr),value :: h
            integer(c_int),value :: penalty, nout
            real(c_double),value :: lambda_lo, lambda_hi
            real(c_double),intent(out) :: lambda, out(*), trace(*)
            integer(c_int64_t),value :: trace_cap
            integer(c_int64_t),intent(out) :: ntrace
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_fit_select_smoothing_reml
        function c_fit_prepare_variance(h,out,nout,ierror) bind(C,name='splpak_b200_fit_prepare_variance') result(rc)
            import :: c_int, c_double, c_ptr
            type(c_ptr),value :: h
            integer(c_int),value :: nout
            real(c_double),intent(out) :: out(*)
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_fit_prepare_variance
        function c_fit_variance(h,x,l1x,nq,nderiv,out,ierror) bind(C,name='splpak_b200_fit_variance') result(rc)
            import :: c_int, c_int64_t, c_ptr, cwp
            type(c_ptr),value :: h
            real(cwp),intent(in) :: x(*)
            integer(c_int),value :: l1x
            integer(c_int64_t),value :: nq
            type(c_ptr),value :: nderiv                      !! c_null_ptr => values
            real(cwp) :: out(*)
            integer(c_int),intent(out) :: ierror
            integer(c_int) :: rc
        end function c_fit_variance
        function c_fit_destroy(h) bind(C,name='splpak_b200_fit_destroy') result(rc)
            import :: c_int, c_ptr
            type(c_ptr),value :: h
            integer(c_int) :: rc
        end function c_fit_destroy
        function c_strerror(code,evaluation) bind(C,name='splpak_b200_strerror') result(p)
            import :: c_int, c_ptr
            integer(c_int),value :: code, evaluation
            type(c_ptr) :: p
        end function c_strerror
    end interface

    contains

    !> cfaerr of the reference (src/splpak.F90:399-407): ' IERR=' I5, then the message.
    subroutine cfaerr(ierr,evaluation)
        integer,intent(in) :: ierr
        logical,intent(in) :: evaluation
        character(kind=c_char),pointer :: s(:)
        type(c_ptr) :: p
        integer :: n
        if (ierr == 0) return
        write (output_unit,'(A,I5)') ' IERR=', ierr
        p = c_strerror(int(ierr,c_int), merge(1_c_int,0_c_int,evaluation))
        call c_f_pointer(p, s, [200])
        n = 0
        do while (n < 200)
            if (s(n+1) == c_null_char) exit
            n = n + 1
        end do
        write (output_unit,'(200A1)') s(1:n)
    end subroutine cfaerr

    subroutine destroy_splpak(me,ndim)
        class(splpak_type),intent(inout) :: me
        integer,intent(in),optional :: ndim
        integer(c_int) :: rc
        if (c_associated(me%handle)) then
            rc = c_fit_destroy(me%handle)
            me%handle = c_null_ptr
        end if
        me%mdim = 0
    end subroutine destroy_splpak

    subroutine splcc(me,ndim,xdata,l1xdat,ydata,ndata,xmin,xmax,nodes,xtrap,coef,ncf,work,nwrk,ierror)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: ndim, l1xdat, ncf, nwrk, ndata
        real(wp),intent(in) :: xdata(l1xdat,ndata), ydata(ndata), xmin(ndim), xmax(ndim), xtrap
        integer,intent(in) :: nodes(ndim)
        real(wp) :: work(nwrk)
        real(wp),intent(out) :: coef(ncf)
        integer,intent(out) :: ierror
        integer(c_int) :: rc, ie
        me%mdim = ndim
        rc = c_splcc(int(ndim,c_int),xdata,int(l1xdat,c_int),ydata,int(ndata,c_int64_t),xmin,xmax,nodes, &
                     xtrap,coef,int(ncf,c_int64_t),work,int(nwrk,c_int64_t),ie)
        ierror = ie
        call cfaerr(ierror,.false.)
    end subroutine splcc

    subroutine splcw(me,ndim,xdata,l1xdat,ydata,wdata,ndata,xmin,xmax,nodes,xtrap,coef,ncf,work,nwrk,ierror)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: ndim, l1xdat, ncf, nwrk, ndata
        real(wp),intent(in) :: xdata(l1xdat,ndata), ydata(ndata), xmin(ndim), xmax(ndim), xtrap
        real(wp),intent(in) :: wdata(:)    !! assumed shape as in the reference (:560); copied if not contiguous
        integer,intent(in) :: nodes(ndim)
        real(wp) :: work(nwrk)
        real(wp),intent(out) :: coef(ncf)
        integer,intent(out) :: ierror
        real(wp),allocatable :: wc(:)
        integer(c_int) :: rc, ie
        me%mdim = ndim
        wc = wdata                         ! contiguous copy (wdata may be a strided section, or size 1 with wdata(1)<0)
        rc = c_splcw(int(ndim,c_int),xdata,int(l1xdat,c_int),ydata,wc,int(ndata,c_int64_t),xmin,xmax,nodes, &
                     xtrap,coef,int(ncf,c_int64_t),work,int(nwrk,c_int64_t),ie)
        ierror = ie
        call cfaerr(ierror,.false.)
    end subroutine splcw

    function splde(me,ndim,x,nderiv,coef,xmin,xmax,nodes,ierror)
        class(splpak_type),intent(inout) :: me
        real(wp) :: splde
        integer,intent(in) :: ndim
        real(wp),intent(in) :: x(ndim), xmin(ndim), xmax(ndim)
        real(wp),intent(in) :: coef(*)     !! intent(out) in the reference although only read (:1103)
        integer,intent(in) :: nderiv(ndim), nodes(ndim)
        integer,intent(out) :: ierror
        integer(c_int) :: ie
        me%mdim = ndim
        splde = c_splde(int(ndim,c_int),x,nderiv,coef,xmin,xmax,nodes,ie)
        ierror = ie
        call cfaerr(ierror,.true.)
    end function splde

    function splfe(me,ndim,x,coef,xmin,xmax,nodes,ierror)
        class(splpak_type),intent(inout) :: me
        real(wp) :: splfe
        integer,intent(in) :: ndim
        real(wp),intent(in) :: x(ndim), xmin(ndim), xmax(ndim)
        real(wp),intent(in) :: coef(*)
        integer,intent(in) :: nodes(ndim)
        integer,intent(out) :: ierror
        integer(c_int) :: ie
        me%mdim = ndim
        splfe = c_splfe(int(ndim,c_int),x,coef,xmin,xmax,nodes,ie)
        ierror = ie
        call cfaerr(ierror,.true.)
    end function splfe

    !> (new) nq points x(l1x,nq) at once; nderiv absent => splfe.
    subroutine evaluate_batch(me,ndim,x,l1x,nq,coef,xmin,xmax,nodes,f,ierror,nderiv)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: ndim, l1x
        integer(int64),intent(in) :: nq
        real(wp),intent(in) :: x(l1x,nq), coef(*), xmin(ndim), xmax(ndim)
        integer,intent(in) :: nodes(ndim)
        real(wp),intent(out) :: f(nq)
        integer,intent(out) :: ierror
        integer,intent(in),optional,target :: nderiv(ndim)
        integer(c_int) :: rc, ie
        type(c_ptr) :: pn
        pn = c_null_ptr
        if (present(nderiv)) pn = c_loc(nderiv)
        rc = c_eval(int(ndim,c_int),x,int(l1x,c_int),int(nq,c_int64_t),pn,coef,xmin,xmax,nodes,f,ie)
        ierror = ie
        call cfaerr(ierror,.true.)
    end subroutine evaluate_batch

    !> (new) every partial derivative up to total order `order` (1 or 2) at nq points x(l1x,nq) in one pass:
    !> f(ncomp,nq) with ncomp = ndim+1 (order 1: the value, d/dx1 .. d/dxn) or (ndim+1)*(ndim+2)/2 (order 2: then
    !> d2/dxi dxj for i <= j in row order).  Component k equals evaluate_batch with the nderiv it names, bit for bit.
    !> An order other than 1 or 2 sets ierror = 104 and leaves f unchanged.
    subroutine evaluate_derivs(me,ndim,x,l1x,nq,order,coef,xmin,xmax,nodes,f,ierror)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: ndim, l1x, order
        integer(int64),intent(in) :: nq
        real(wp),intent(in) :: x(l1x,nq), coef(*), xmin(ndim), xmax(ndim)
        integer,intent(in) :: nodes(ndim)
        real(wp),intent(inout) :: f(*)
        integer,intent(out) :: ierror
        integer(c_int) :: rc, ie
        rc = c_eval_derivs(int(ndim,c_int),x,int(l1x,c_int),int(nq,c_int64_t),int(order,c_int),coef,xmin,xmax,nodes,f,ie)
        ierror = ie
        call cfaerr(ierror,.true.)
    end subroutine evaluate_derivs

    !> (new) value or partial derivative on the tensor grid spanned by the ndim axes stored one after the other in
    !> `axes` (axis d has naxis(d) points); f(naxis(1),...,naxis(ndim)); nderiv absent => splfe.
    subroutine evaluate_grid(me,ndim,axes,naxis,coef,xmin,xmax,nodes,f,ierror,nderiv)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: ndim
        integer(int64),intent(in) :: naxis(ndim)
        real(wp),intent(in) :: axes(*), coef(*), xmin(ndim), xmax(ndim)
        integer,intent(in) :: nodes(ndim)
        real(wp),intent(out) :: f(*)
        integer,intent(out) :: ierror
        integer,intent(in),optional,target :: nderiv(ndim)
        integer(c_int) :: rc, ie
        type(c_ptr) :: pn
        pn = c_null_ptr
        if (present(nderiv)) pn = c_loc(nderiv)
        rc = c_eval_grid(int(ndim,c_int),axes,naxis,pn,coef,xmin,xmax,nodes,f,ie)
        ierror = ie
        call cfaerr(ierror,.true.)
    end subroutine evaluate_grid

    !> (new) streaming fit: validates the grid like splcw (101,102,103) and allocates device buffers.
    subroutine create(me,ndim,xmin,xmax,nodes,xtrap,ierror)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: ndim
        real(wp),intent(in) :: xmin(ndim), xmax(ndim), xtrap
        integer,intent(in) :: nodes(ndim)
        integer,intent(out) :: ierror
        integer(c_int) :: rc, ie
        call me%destroy()
        me%mdim = ndim
        rc = c_fit_create(int(ndim,c_int),xmin,xmax,nodes,xtrap,me%handle,ie)
        ierror = ie
        call cfaerr(ierror,.false.)
    end subroutine create

    !> (new) choose the solver of a streaming fit, after create and before the first add_points:
    !  0 = band Cholesky of the normal equations (default), 1 = Householder reductions only, like the
    !  reference's suprls (accurate at cond(A); 1-D..3-D).  ierror = 203 when not available.
    subroutine set_solver(me,solver,ierror)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: solver
        integer,intent(out) :: ierror
        ierror = int(c_fit_set_solver(me%handle,int(solver,c_int)))
    end subroutine set_solver

    !> (new) smoothing of a streaming fit, after create and before compute: the Cholesky fit adds
    !  lambda * the integral over [xmin, xmax] of the penalty to the least-squares objective.
    !  penalty 0 = sum of squared second derivatives (curvature), 1 = thin plate (mixed ones too).
    !  lambda = 0 (default) is the unsmoothed fit.  ierror = 203 for lambda < 0 or not finite, an
    !  unknown penalty, or lambda > 0 with the orthogonal solver.
    subroutine set_smoothing(me,lambda,penalty,ierror)
        class(splpak_type),intent(inout) :: me
        real(c_double),intent(in) :: lambda
        integer,intent(in) :: penalty
        integer,intent(out) :: ierror
        ierror = int(c_fit_set_smoothing(me%handle,lambda,int(penalty,c_int)))
    end subroutine set_smoothing

    !> (new) generalized cross-validation: call before the first add_points (ierror = 203 otherwise,
    !  or with the orthogonal solver).  Persists across reset.
    subroutine enable_gcv(me,ierror)
        class(splpak_type),intent(inout) :: me
        integer,intent(out) :: ierror
        ierror = int(c_fit_enable_gcv(me%handle))
    end subroutine enable_gcv

    !> (new) GCV score of smoothing lambda after the assembly, before compute (changes nothing compute
    !  sees): score = [V, RSS, edf, N, ywy].  ierror = 107 for a non-positive pivot, 203 when refused.
    subroutine smoothing_score(me,lambda,penalty,score,ierror)
        class(splpak_type),intent(inout) :: me
        real(c_double),intent(in) :: lambda
        integer,intent(in) :: penalty
        real(c_double),intent(out) :: score(5)
        integer,intent(out) :: ierror
        integer(c_int) :: ierr, rc
        rc = c_fit_smoothing_score(me%handle,lambda,int(penalty,c_int),score,5_c_int,ierr)
        ierror = int(rc)
    end subroutine smoothing_score

    !> (new) lambda minimising the GCV score over [lambda_lo, lambda_hi] (either <= 0: the default range),
    !  then set on the fit, so the next compute is the selected fit.  score as smoothing_score.
    subroutine select_smoothing(me,penalty,lambda_lo,lambda_hi,lambda,score,ierror)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: penalty
        real(c_double),intent(in) :: lambda_lo, lambda_hi
        real(c_double),intent(out) :: lambda, score(5)
        integer,intent(out) :: ierror
        integer(c_int) :: ierr, rc
        integer(c_int64_t) :: ntrace
        real(c_double) :: trace(4)
        rc = c_fit_select_smoothing(me%handle,int(penalty,c_int),lambda_lo,lambda_hi,lambda,score,5_c_int, &
                                    trace,0_c_int64_t,ntrace,ierr)
        ierror = int(rc)
    end subroutine select_smoothing

    !> (new) REML score of smoothing lambda > 0 after the assembly, before compute (changes nothing compute
    !  sees): score = [V_R, D_p, log|M|, n, ywy, phi], n counting the constraint rows, phi = D_p / (n - Mp).
    !  ierror = 107 for a non-positive pivot, 203 when refused (also for lambda <= 0).
    subroutine reml_score(me,lambda,penalty,score,ierror)
        class(splpak_type),intent(inout) :: me
        real(c_double),intent(in) :: lambda
        integer,intent(in) :: penalty
        real(c_double),intent(out) :: score(6)
        integer,intent(out) :: ierror
        integer(c_int) :: ierr, rc
        rc = c_fit_reml_score(me%handle,lambda,int(penalty,c_int),score,6_c_int,ierr)
        ierror = int(rc)
    end subroutine reml_score

    !> (new) lambda minimising the REML score over [lambda_lo, lambda_hi] (either <= 0: the default range),
    !  then set on the fit, so the next compute is the selected fit.  score as reml_score.
    subroutine select_smoothing_reml(me,penalty,lambda_lo,lambda_hi,lambda,score,ierror)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: penalty
        real(c_double),intent(in) :: lambda_lo, lambda_hi
        real(c_double),intent(out) :: lambda, score(6)
        integer,intent(out) :: ierror
        integer(c_int) :: ierr, rc
        integer(c_int64_t) :: ntrace
        real(c_double) :: trace(4)
        rc = c_fit_select_smoothing_reml(me%handle,int(penalty,c_int),lambda_lo,lambda_hi,lambda,score,6_c_int, &
                                         trace,0_c_int64_t,ntrace,ierr)
        ierror = int(rc)
    end subroutine select_smoothing_reml

    !> (new) posterior variances of a smoothing fit, after the assembly (and select_smoothing) and before
    !  compute: builds the per-window tables from Sigma of the fit's current lambda (scoring once unless
    !  select_smoothing left that Sigma behind).  score = [V, RSS, edf, N, ywy, sigma2], sigma2 = RSS / (N - edf).
    !  ierror = 203 when refused (GCV not enabled, orthogonal solver, after compute), 204 allocation, 107 pivot.
    subroutine prepare_variance(me,score,ierror)
        class(splpak_type),intent(inout) :: me
        real(c_double),intent(out) :: score(6)
        integer,intent(out) :: ierror
        integer(c_int) :: ierr, rc
        rc = c_fit_prepare_variance(me%handle,score,6_c_int,ierr)
        ierror = int(rc)
    end subroutine prepare_variance

    !> (new) q(i) = b(x_i)^T Sigma b(x_i) at the nq points x(:,i), after prepare_variance (any time, also after
    !  compute): the posterior variance of the fitted value -- of the partial derivative nderiv when present --
    !  divided by sigma2.  ierror = 203 without valid tables, 104 for nderiv outside 0..2.
    subroutine variance(me,x,l1x,nq,q,ierror,nderiv)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: l1x
        integer(int64),intent(in) :: nq
        real(wp),intent(in) :: x(l1x,nq)
        real(wp),intent(out) :: q(nq)
        integer,intent(out) :: ierror
        integer,intent(in),optional,target :: nderiv(me%mdim)
        integer(c_int) :: rc, ie
        type(c_ptr) :: pn
        pn = c_null_ptr
        if (present(nderiv)) pn = c_loc(nderiv)
        rc = c_fit_variance(me%handle,x,int(l1x,c_int),int(nq,c_int64_t),pn,q,ie)
        ierror = int(rc)
    end subroutine variance

    !> (new) accumulate n more points; wdata absent (or wdata(1)<0) => all weights 1.
    subroutine add_points(me,xdata,l1xdat,ydata,ndata,ierror,wdata)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: l1xdat
        integer(int64),intent(in) :: ndata
        real(wp),intent(in) :: xdata(l1xdat,ndata), ydata(ndata)
        integer,intent(out) :: ierror
        real(wp),intent(in),optional :: wdata(ndata)
        integer(c_int) :: weighted
        real(wp) :: dummy(1)
        weighted = 0
        if (present(wdata)) then
            if (wdata(1) >= 0.0_wp) weighted = 1
            ierror = c_fit_add_points(me%handle,xdata,int(l1xdat,c_int),ydata,wdata,weighted,int(ndata,c_int64_t))
        else
            dummy = -1.0_wp
            ierror = c_fit_add_points(me%handle,xdata,int(l1xdat,c_int),ydata,dummy,weighted,int(ndata,c_int64_t))
        end if
        call cfaerr(ierror,.false.)
    end subroutine add_points

    !> (new) add the data-sparse constraint rows, factor, solve; codes 104/106/107 as splcw.
    subroutine compute(me,coef,ncf,nwrk,ierror)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: ncf, nwrk
        real(wp),intent(out) :: coef(ncf)
        integer,intent(out) :: ierror
        integer(c_int) :: rc, ie
        rc = c_fit_compute(me%handle,coef,int(ncf,c_int64_t),int(nwrk,c_int64_t),ie)
        ierror = ie
        call cfaerr(ierror,.false.)
    end subroutine compute

    !> (new) one step of corrected-semi-normal-equations refinement after `compute`, with the SAME points
    !> (initialize => splcc/splcw do this by themselves when derivative-constraint rows fired).
    subroutine refine(me,xdata,l1xdat,ydata,ndata,coef,ncf,ierror,wdata)
        class(splpak_type),intent(inout) :: me
        integer,intent(in) :: l1xdat, ncf
        integer(int64),intent(in) :: ndata
        real(wp),intent(in) :: xdata(l1xdat,ndata), ydata(ndata)
        real(wp),intent(out) :: coef(ncf)
        integer,intent(out) :: ierror
        real(wp),intent(in),optional :: wdata(ndata)
        integer(c_int) :: weighted, rc, ie
        real(wp) :: dummy(1)
        ierror = c_fit_refine_begin(me%handle)
        if (ierror /= 0) then
            call cfaerr(ierror,.false.)
            return
        end if
        weighted = 0
        if (present(wdata)) then
            if (wdata(1) >= 0.0_wp) weighted = 1
            ierror = c_fit_refine_add_points(me%handle,xdata,int(l1xdat,c_int),ydata,wdata,weighted,int(ndata,c_int64_t))
        else
            dummy = -1.0_wp
            ierror = c_fit_refine_add_points(me%handle,xdata,int(l1xdat,c_int),ydata,dummy,weighted,int(ndata,c_int64_t))
        end if
        if (ierror == 0) then
            rc = c_fit_refine_compute(me%handle,coef,int(ncf,c_int64_t),ie)
            ierror = ie
        end if
        call cfaerr(ierror,.false.)
    end subroutine refine

    end module splpak_module
