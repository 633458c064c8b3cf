!!
!! NKA_B200_C -- ISO_C_BINDING interfaces to libnka_b200.so
!!
!! One interface block per C entry point of include/nonlinear_krylov_accelerator.h and
!! include/nka_b200.h.  Pure declarations: no executable code.  The three nka_type
!! modules in this directory (F95/, F08/, F08-vector/) are thin layers over these.
!!
!! NOT COMPILED in the build image (it has no Fortran compiler).  Standard F2003
!! interoperability only; every symbol below is exercised with the same argument
!! passing (scalars by value, arrays by address) by tests/test_fortran_abi.py.
!!

module nka_b200_c

  use, intrinsic :: iso_c_binding
  implicit none
  public

  !! include/nka_b200.h: nka_stop_test, the stopping rule of nka_batch_loop_create_stop and
  !! nka_batch_queue_create_stop.  The *_dev components are device addresses (c_null_ptr: the scalar
  !! applies; scale_dev c_null_ptr: no scale).  Declare it with the target attribute and pass c_loc of it.
  type, bind(C) :: nka_stop_test
    real(c_double) :: atol, rtol, dtol
    integer(c_int) :: maxit
    type(c_ptr) :: atol_dev, rtol_dev, maxit_dev, scale_dev
    integer(c_size_t) :: ldscale
  end type nka_stop_test

  interface

    !! NKA nka_init_ex (size_t vlen, int mvec, double vtol, int device, void *stream)
    function nka_init_ex(vlen, mvec, vtol, device, stream) bind(C, name='nka_init_ex') result(handle)
      import :: c_ptr, c_size_t, c_int, c_double
      integer(c_size_t), value :: vlen
      integer(c_int),    value :: mvec
      real(c_double),    value :: vtol
      integer(c_int),    value :: device
      type(c_ptr),       value :: stream
      type(c_ptr) :: handle
    end function

    !! void nka_delete (NKA)
    subroutine nka_delete_c(handle) bind(C, name='nka_delete')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    !! void nka_accel_update (NKA, double *f) -- f host or device, detected by the library
    subroutine nka_accel_update_c(handle, f) bind(C, name='nka_accel_update')
      import :: c_ptr, c_double
      type(c_ptr), value :: handle
      real(c_double), intent(inout) :: f(*)
    end subroutine

    !! void nka_accel_update_host (NKA, double *f_host)
    subroutine nka_accel_update_host(handle, f) bind(C, name='nka_accel_update_host')
      import :: c_ptr, c_double
      type(c_ptr), value :: handle
      real(c_double), intent(inout) :: f(*)
    end subroutine

    !! void nka_accel_update_dev (NKA, double *f_dev) -- f is a device address held in a c_ptr
    subroutine nka_accel_update_dev(handle, f_dev) bind(C, name='nka_accel_update_dev')
      import :: c_ptr
      type(c_ptr), value :: handle
      type(c_ptr), value :: f_dev
    end subroutine

    subroutine nka_restart_c(handle) bind(C, name='nka_restart')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    subroutine nka_relax_c(handle) bind(C, name='nka_relax')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    function nka_num_vec_c(handle) bind(C, name='nka_num_vec') result(n)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int) :: n
    end function

    function nka_max_vec_c(handle) bind(C, name='nka_max_vec') result(n)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int) :: n
    end function

    function nka_vec_len_c(handle) bind(C, name='nka_vec_len') result(n)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int) :: n
    end function

    function nka_vec_len64(handle) bind(C, name='nka_vec_len64') result(n)
      import :: c_ptr, c_size_t
      type(c_ptr), value :: handle
      integer(c_size_t) :: n
    end function

    function nka_vec_tol_c(handle) bind(C, name='nka_vec_tol') result(vtol)
      import :: c_ptr, c_double
      type(c_ptr), value :: handle
      real(c_double) :: vtol
    end function

    subroutine nka_set_vec_tol_c(handle, vtol) bind(C, name='nka_set_vec_tol')
      import :: c_ptr, c_double
      type(c_ptr), value :: handle
      real(c_double), value :: vtol
    end subroutine

    !! void nka_set_dot_prod_ctx (NKA, double (*dp)(int, double *, double *, void *), void *ctx)
    !! dp = c_funloc of a bind(C) trampoline, ctx = whatever it needs to find the user's procedure
    !! pointer; c_null_funptr restores the built-in reductions.
    subroutine nka_set_dot_prod_ctx(handle, dp, ctx) bind(C, name='nka_set_dot_prod_ctx')
      import :: c_ptr, c_funptr
      type(c_ptr), value :: handle
      type(c_funptr), value :: dp
      type(c_ptr), value :: ctx
    end subroutine

    function nka_defined_c(handle) bind(C, name='nka_defined') result(ok)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int) :: ok
    end function

    subroutine nka_set_stream(handle, stream) bind(C, name='nka_set_stream')
      import :: c_ptr
      type(c_ptr), value :: handle, stream
    end subroutine

    subroutine nka_synchronize(handle) bind(C, name='nka_synchronize')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    !! int nka_comm_unique_id (void *id128) ; int nka_comm_init (NKA, int nranks, int rank, const void *id128)
    function nka_comm_unique_id(id128) bind(C, name='nka_comm_unique_id') result(rc)
      import :: c_int, c_char
      character(kind=c_char), intent(out) :: id128(128)
      integer(c_int) :: rc
    end function

    function nka_comm_init(handle, nranks, rank, id128) bind(C, name='nka_comm_init') result(rc)
      import :: c_ptr, c_int, c_char
      type(c_ptr), value :: handle
      integer(c_int), value :: nranks, rank
      character(kind=c_char), intent(in) :: id128(128)
      integer(c_int) :: rc
    end function

    !! ---- device vectors (gpu_vector) ----

    function nka_vec_create(n, device, stream) bind(C, name='nka_vec_create') result(v)
      import :: c_ptr, c_size_t, c_int
      integer(c_size_t), value :: n
      integer(c_int),    value :: device
      type(c_ptr),       value :: stream
      type(c_ptr) :: v
    end function

    function nka_vec_clone(src) bind(C, name='nka_vec_clone') result(v)
      import :: c_ptr
      type(c_ptr), value :: src
      type(c_ptr) :: v
    end function

    subroutine nka_vec_destroy(v) bind(C, name='nka_vec_destroy')
      import :: c_ptr
      type(c_ptr), value :: v
    end subroutine

    function nka_vec_size(v) bind(C, name='nka_vec_size') result(n)
      import :: c_ptr, c_size_t
      type(c_ptr), value :: v
      integer(c_size_t) :: n
    end function

    function nka_vec_data(v) bind(C, name='nka_vec_data') result(dptr)
      import :: c_ptr
      type(c_ptr), value :: v
      type(c_ptr) :: dptr
    end function

    subroutine nka_vec_set_host(v, host) bind(C, name='nka_vec_set_host')
      import :: c_ptr, c_double
      type(c_ptr), value :: v
      real(c_double), intent(in) :: host(*)
    end subroutine

    subroutine nka_vec_get_host(v, host) bind(C, name='nka_vec_get_host')
      import :: c_ptr, c_double
      type(c_ptr), value :: v
      real(c_double), intent(out) :: host(*)
    end subroutine

    subroutine nka_vec_copy(dst, src) bind(C, name='nka_vec_copy')
      import :: c_ptr
      type(c_ptr), value :: dst, src
    end subroutine

    subroutine nka_vec_setval(v, val) bind(C, name='nka_vec_setval')
      import :: c_ptr, c_double
      type(c_ptr), value :: v
      real(c_double), value :: val
    end subroutine

    subroutine nka_vec_scale(v, a) bind(C, name='nka_vec_scale')
      import :: c_ptr, c_double
      type(c_ptr), value :: v
      real(c_double), value :: a
    end subroutine

    subroutine nka_vec_update1(y, a, x) bind(C, name='nka_vec_update1')
      import :: c_ptr, c_double
      type(c_ptr), value :: y, x
      real(c_double), value :: a
    end subroutine

    subroutine nka_vec_update2(y, a, x, b) bind(C, name='nka_vec_update2')
      import :: c_ptr, c_double
      type(c_ptr), value :: y, x
      real(c_double), value :: a, b
    end subroutine

    subroutine nka_vec_update3(z, a, x, b, y) bind(C, name='nka_vec_update3')
      import :: c_ptr, c_double
      type(c_ptr), value :: z, x, y
      real(c_double), value :: a, b
    end subroutine

    subroutine nka_vec_update4(z, a, x, b, y, c) bind(C, name='nka_vec_update4')
      import :: c_ptr, c_double
      type(c_ptr), value :: z, x, y
      real(c_double), value :: a, b, c
    end subroutine

    function nka_vec_dot(x, y) bind(C, name='nka_vec_dot') result(dp)
      import :: c_ptr, c_double
      type(c_ptr), value :: x, y
      real(c_double) :: dp
    end function

    function nka_vec_norm2(x) bind(C, name='nka_vec_norm2') result(nrm)
      import :: c_ptr, c_double
      type(c_ptr), value :: x
      real(c_double) :: nrm
    end function

    function nka_vec_comm_init(v, nranks, rank, id128) bind(C, name='nka_vec_comm_init') result(rc)
      import :: c_ptr, c_int, c_char
      type(c_ptr), value :: v
      integer(c_int), value :: nranks, rank
      character(kind=c_char), intent(in) :: id128(128)
      integer(c_int) :: rc
    end function

    function nka_init_like(proto, mvec, vtol) bind(C, name='nka_init_like') result(handle)
      import :: c_ptr, c_int, c_double
      type(c_ptr), value :: proto
      integer(c_int), value :: mvec
      real(c_double), value :: vtol
      type(c_ptr) :: handle
    end function

    subroutine nka_accel_update_vec(handle, f) bind(C, name='nka_accel_update_vec')
      import :: c_ptr
      type(c_ptr), value :: handle, f
    end subroutine

    !! ---- batched accelerators (include/nka_b200.h): the handle is a struct nka_batch * in a c_ptr

    !! NKABATCH nka_batch_init (int nbatch, size_t vlen, int mvec, double vtol, int device, void *stream)
    function nka_batch_init(nbatch, vlen, mvec, vtol, device, stream) bind(C, name='nka_batch_init') result(handle)
      import :: c_ptr, c_size_t, c_int, c_double
      integer(c_int),    value :: nbatch
      integer(c_size_t), value :: vlen
      integer(c_int),    value :: mvec
      real(c_double),    value :: vtol
      integer(c_int),    value :: device
      type(c_ptr),       value :: stream
      type(c_ptr) :: handle
    end function

    subroutine nka_batch_delete(handle) bind(C, name='nka_batch_delete')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    !! void nka_batch_accel_update (NKABATCH, double *f_dev, size_t ldf, const unsigned char *active_dev)
    !! f_dev: the device array of nbatch rows (CUDA Fortran: a device array, passed by address);
    !! active_dev: c_null_ptr or the device address of nbatch bytes
    subroutine nka_batch_accel_update(handle, f_dev, ldf, active_dev) bind(C, name='nka_batch_accel_update')
      import :: c_ptr, c_double, c_size_t
      type(c_ptr), value :: handle
      real(c_double), intent(inout) :: f_dev(*)
      integer(c_size_t), value :: ldf
      type(c_ptr), value :: active_dev
    end subroutine

    subroutine nka_batch_relax(handle, mask_dev) bind(C, name='nka_batch_relax')
      import :: c_ptr
      type(c_ptr), value :: handle, mask_dev
    end subroutine

    subroutine nka_batch_restart(handle, mask_dev) bind(C, name='nka_batch_restart')
      import :: c_ptr
      type(c_ptr), value :: handle, mask_dev
    end subroutine

    subroutine nka_batch_set_vec_tol(handle, vtol) bind(C, name='nka_batch_set_vec_tol')
      import :: c_ptr, c_double
      type(c_ptr), value :: handle
      real(c_double), value :: vtol
    end subroutine

    !! out: c_loc of an integer(c_int) array of nbatch elements on the host
    subroutine nka_batch_num_vec(handle, out) bind(C, name='nka_batch_num_vec')
      import :: c_ptr
      type(c_ptr), value :: handle, out
    end subroutine

    function nka_batch_defined(handle) bind(C, name='nka_batch_defined') result(ok)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int) :: ok
    end function

    !! out: c_loc of an nka_state_view on the host
    subroutine nka_batch_get_state(handle, member, out) bind(C, name='nka_batch_get_state')
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int), value :: member
      type(c_ptr), value :: out
    end subroutine

    subroutine nka_batch_set_stream(handle, stream) bind(C, name='nka_batch_set_stream')
      import :: c_ptr
      type(c_ptr), value :: handle, stream
    end subroutine

    subroutine nka_batch_synchronize(handle) bind(C, name='nka_batch_synchronize')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    function nka_batch_stream_capturing(handle) bind(C, name='nka_batch_stream_capturing') result(c)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int) :: c
    end function

    function nka_batch_launch_count(handle) bind(C, name='nka_batch_launch_count') result(n)
      import :: c_ptr, c_long_long
      type(c_ptr), value :: handle
      integer(c_long_long) :: n
    end function

    !! ---- device-side fixed-point loops (include/nka_b200.h): the handle is a struct nka_batch_loop *

    !! NKABATCHLOOP nka_batch_loop_create (NKABATCH, void *residual_graph, double *x_dev, size_t ldx,
    !!                                     double *f_dev, size_t ldf, double atol, double rtol, int maxit)
    !! residual_graph: a cudaGraph_t; x_dev, f_dev: device arrays of nbatch rows, passed as
    !! nka_batch_accel_update's f_dev is.  c_null_ptr if CUDA refuses the graph.
    function nka_batch_loop_create(batch, residual_graph, x_dev, ldx, f_dev, ldf, atol, rtol, maxit) &
        bind(C, name='nka_batch_loop_create') result(handle)
      import :: c_ptr, c_double, c_size_t, c_int
      type(c_ptr), value :: batch, residual_graph
      real(c_double), intent(inout) :: x_dev(*)
      integer(c_size_t), value :: ldx
      real(c_double), intent(inout) :: f_dev(*)
      integer(c_size_t), value :: ldf
      real(c_double), value :: atol, rtol
      integer(c_int), value :: maxit
      type(c_ptr) :: handle
    end function

    subroutine nka_batch_loop_launch(handle) bind(C, name='nka_batch_loop_launch')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    !! iters, status: c_loc of integer(c_int) arrays of nbatch elements on the host; norm: nbatch reals
    subroutine nka_batch_loop_results(handle, iters, status, norm) bind(C, name='nka_batch_loop_results')
      import :: c_ptr, c_double
      type(c_ptr), value :: handle, iters, status
      real(c_double), intent(out) :: norm(*)
    end subroutine

    !! norms: (maxit+1) x nbatch reals on the host, member index fastest
    subroutine nka_batch_loop_history(handle, norms) bind(C, name='nka_batch_loop_history')
      import :: c_ptr, c_double
      type(c_ptr), value :: handle
      real(c_double), intent(out) :: norms(*)
    end subroutine

    subroutine nka_batch_loop_destroy(handle) bind(C, name='nka_batch_loop_destroy')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    !! ---- device-side work queues (include/nka_b200.h): the handle is a struct nka_batch_queue *

    !! NKABATCHQUEUE nka_batch_queue_create (NKABATCH, void *residual_graph, double *x_dev, size_t ldx,
    !!     double *f_dev, size_t ldf, int *slot_problem_dev, const double *x0_dev, size_t ldx0,
    !!     double *xout_dev, size_t ldxout, size_t nproblems, double atol, double rtol, int maxit)
    !! x_dev, f_dev: nbatch rows; x0_dev, xout_dev: nproblems rows, passed as nka_batch_accel_update's
    !! f_dev is; slot_problem_dev: the device address of nbatch integer(c_int).  c_null_ptr if CUDA
    !! refuses the graph.
    function nka_batch_queue_create(batch, residual_graph, x_dev, ldx, f_dev, ldf, slot_problem_dev, x0_dev, ldx0, &
                                    xout_dev, ldxout, nproblems, atol, rtol, maxit) &
        bind(C, name='nka_batch_queue_create') result(handle)
      import :: c_ptr, c_double, c_size_t, c_int
      type(c_ptr), value :: batch, residual_graph
      real(c_double), intent(inout) :: x_dev(*)
      integer(c_size_t), value :: ldx
      real(c_double), intent(inout) :: f_dev(*)
      integer(c_size_t), value :: ldf
      type(c_ptr), value :: slot_problem_dev
      real(c_double), intent(in) :: x0_dev(*)
      integer(c_size_t), value :: ldx0
      real(c_double), intent(inout) :: xout_dev(*)
      integer(c_size_t), value :: ldxout, nproblems
      real(c_double), value :: atol, rtol
      integer(c_int), value :: maxit
      type(c_ptr) :: handle
    end function

    subroutine nka_batch_queue_launch(handle) bind(C, name='nka_batch_queue_launch')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    !! iters, status: c_loc of integer(c_int) arrays of nproblems elements on the host; norm: nproblems reals
    subroutine nka_batch_queue_results(handle, iters, status, norm) bind(C, name='nka_batch_queue_results')
      import :: c_ptr, c_double
      type(c_ptr), value :: handle, iters, status
      real(c_double), intent(out) :: norm(*)
    end subroutine

    subroutine nka_batch_queue_destroy(handle) bind(C, name='nka_batch_queue_destroy')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    !! ---- per-problem stopping tests (include/nka_b200.h): the creates above with an nka_stop_test

    !! NKABATCHLOOP nka_batch_loop_create_stop (NKABATCH, void *residual_graph, double *x_dev, size_t ldx,
    !!                                          double *f_dev, size_t ldf, const nka_stop_test *stop)
    !! stop: c_loc of a type(nka_stop_test), target.  c_null_ptr if CUDA refuses the graph.
    function nka_batch_loop_create_stop(batch, residual_graph, x_dev, ldx, f_dev, ldf, stop) &
        bind(C, name='nka_batch_loop_create_stop') result(handle)
      import :: c_ptr, c_double, c_size_t
      type(c_ptr), value :: batch, residual_graph
      real(c_double), intent(inout) :: x_dev(*)
      integer(c_size_t), value :: ldx
      real(c_double), intent(inout) :: f_dev(*)
      integer(c_size_t), value :: ldf
      type(c_ptr), value :: stop
      type(c_ptr) :: handle
    end function

    !! NKABATCHQUEUE nka_batch_queue_create_stop (NKABATCH, void *residual_graph, double *x_dev, size_t ldx,
    !!     double *f_dev, size_t ldf, int *slot_problem_dev, const double *x0_dev, size_t ldx0,
    !!     double *xout_dev, size_t ldxout, size_t nproblems, const nka_stop_test *stop)
    !! stop: c_loc of a type(nka_stop_test), target; its arrays hold one entry per problem.
    function nka_batch_queue_create_stop(batch, residual_graph, x_dev, ldx, f_dev, ldf, slot_problem_dev, x0_dev, ldx0, &
                                         xout_dev, ldxout, nproblems, stop) &
        bind(C, name='nka_batch_queue_create_stop') result(handle)
      import :: c_ptr, c_double, c_size_t
      type(c_ptr), value :: batch, residual_graph
      real(c_double), intent(inout) :: x_dev(*)
      integer(c_size_t), value :: ldx
      real(c_double), intent(inout) :: f_dev(*)
      integer(c_size_t), value :: ldf
      type(c_ptr), value :: slot_problem_dev
      real(c_double), intent(in) :: x0_dev(*)
      integer(c_size_t), value :: ldx0
      real(c_double), intent(inout) :: xout_dev(*)
      integer(c_size_t), value :: ldxout, nproblems
      type(c_ptr), value :: stop
      type(c_ptr) :: handle
    end function

    !! ---- residual-growth restarts (include/nka_b200.h): the _stop creates with restart_growth

    !! NKABATCHLOOP nka_batch_loop_create_restart (NKABATCH, void *residual_graph, double *x_dev, size_t ldx,
    !!     double *f_dev, size_t ldf, const nka_stop_test *stop, double restart_growth)
    !! restart_growth: 0 (off) or finite and > 0.  c_null_ptr if CUDA refuses the graph.
    function nka_batch_loop_create_restart(batch, residual_graph, x_dev, ldx, f_dev, ldf, stop, restart_growth) &
        bind(C, name='nka_batch_loop_create_restart') result(handle)
      import :: c_ptr, c_double, c_size_t
      type(c_ptr), value :: batch, residual_graph
      real(c_double), intent(inout) :: x_dev(*)
      integer(c_size_t), value :: ldx
      real(c_double), intent(inout) :: f_dev(*)
      integer(c_size_t), value :: ldf
      type(c_ptr), value :: stop
      real(c_double), value :: restart_growth
      type(c_ptr) :: handle
    end function

    !! NKABATCHQUEUE nka_batch_queue_create_restart (NKABATCH, void *residual_graph, double *x_dev, size_t ldx,
    !!     double *f_dev, size_t ldf, int *slot_problem_dev, const double *x0_dev, size_t ldx0,
    !!     double *xout_dev, size_t ldxout, size_t nproblems, const nka_stop_test *stop, double restart_growth)
    function nka_batch_queue_create_restart(batch, residual_graph, x_dev, ldx, f_dev, ldf, slot_problem_dev, x0_dev, &
                                            ldx0, xout_dev, ldxout, nproblems, stop, restart_growth) &
        bind(C, name='nka_batch_queue_create_restart') result(handle)
      import :: c_ptr, c_double, c_size_t
      type(c_ptr), value :: batch, residual_graph
      real(c_double), intent(inout) :: x_dev(*)
      integer(c_size_t), value :: ldx
      real(c_double), intent(inout) :: f_dev(*)
      integer(c_size_t), value :: ldf
      type(c_ptr), value :: slot_problem_dev
      real(c_double), intent(in) :: x0_dev(*)
      integer(c_size_t), value :: ldx0
      real(c_double), intent(inout) :: xout_dev(*)
      integer(c_size_t), value :: ldxout, nproblems
      type(c_ptr), value :: stop
      real(c_double), value :: restart_growth
      type(c_ptr) :: handle
    end function

    !! restarts: c_loc of an integer(c_int) array of nbatch elements on the host
    subroutine nka_batch_loop_restarts(handle, restarts) bind(C, name='nka_batch_loop_restarts')
      import :: c_ptr
      type(c_ptr), value :: handle, restarts
    end subroutine

    !! restarts: c_loc of an integer(c_int) array of nproblems elements on the host
    subroutine nka_batch_queue_restarts(handle, restarts) bind(C, name='nka_batch_queue_restarts')
      import :: c_ptr
      type(c_ptr), value :: handle, restarts
    end subroutine

    !! ---- interleaved batched accelerators (include/nka_b200.h): the handle is a struct nka_ibatch * in a c_ptr.
    !! A Fortran f(ncell, nvar) with one member per cell is f_dev with ldf = ncell (>= nbatch).

    !! NKAIBATCH nka_ibatch_init (int nbatch, size_t vlen, int mvec, double vtol, int device, void *stream)
    function nka_ibatch_init(nbatch, vlen, mvec, vtol, device, stream) bind(C, name='nka_ibatch_init') result(handle)
      import :: c_ptr, c_size_t, c_int, c_double
      integer(c_int),    value :: nbatch
      integer(c_size_t), value :: vlen
      integer(c_int),    value :: mvec
      real(c_double),    value :: vtol
      integer(c_int),    value :: device
      type(c_ptr),       value :: stream
      type(c_ptr) :: handle
    end function

    subroutine nka_ibatch_delete(handle) bind(C, name='nka_ibatch_delete')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    !! void nka_ibatch_accel_update (NKAIBATCH, double *f_dev, size_t ldf, const unsigned char *active_dev)
    !! f_dev: the device array f(ldf, vlen), element i of member b at f(b, i) (CUDA Fortran: a device array,
    !! passed by address); active_dev: c_null_ptr or the device address of nbatch bytes
    subroutine nka_ibatch_accel_update(handle, f_dev, ldf, active_dev) bind(C, name='nka_ibatch_accel_update')
      import :: c_ptr, c_double, c_size_t
      type(c_ptr), value :: handle
      real(c_double), intent(inout) :: f_dev(*)
      integer(c_size_t), value :: ldf
      type(c_ptr), value :: active_dev
    end subroutine

    subroutine nka_ibatch_relax(handle, mask_dev) bind(C, name='nka_ibatch_relax')
      import :: c_ptr
      type(c_ptr), value :: handle, mask_dev
    end subroutine

    subroutine nka_ibatch_restart(handle, mask_dev) bind(C, name='nka_ibatch_restart')
      import :: c_ptr
      type(c_ptr), value :: handle, mask_dev
    end subroutine

    subroutine nka_ibatch_set_vec_tol(handle, vtol) bind(C, name='nka_ibatch_set_vec_tol')
      import :: c_ptr, c_double
      type(c_ptr), value :: handle
      real(c_double), value :: vtol
    end subroutine

    !! out: c_loc of an integer(c_int) array of nbatch elements on the host
    subroutine nka_ibatch_num_vec(handle, out) bind(C, name='nka_ibatch_num_vec')
      import :: c_ptr
      type(c_ptr), value :: handle, out
    end subroutine

    function nka_ibatch_defined(handle) bind(C, name='nka_ibatch_defined') result(ok)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int) :: ok
    end function

    !! out: c_loc of an nka_state_view on the host
    subroutine nka_ibatch_get_state(handle, member, out) bind(C, name='nka_ibatch_get_state')
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int), value :: member
      type(c_ptr), value :: out
    end subroutine

    subroutine nka_ibatch_set_stream(handle, stream) bind(C, name='nka_ibatch_set_stream')
      import :: c_ptr
      type(c_ptr), value :: handle, stream
    end subroutine

    subroutine nka_ibatch_synchronize(handle) bind(C, name='nka_ibatch_synchronize')
      import :: c_ptr
      type(c_ptr), value :: handle
    end subroutine

    function nka_ibatch_stream_capturing(handle) bind(C, name='nka_ibatch_stream_capturing') result(c)
      import :: c_ptr, c_int
      type(c_ptr), value :: handle
      integer(c_int) :: c
    end function

    function nka_ibatch_launch_count(handle) bind(C, name='nka_ibatch_launch_count') result(n)
      import :: c_ptr, c_long_long
      type(c_ptr), value :: handle
      integer(c_long_long) :: n
    end function

  end interface

end module nka_b200_c
