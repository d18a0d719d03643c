! ISO_C_BINDING interface to libunconfined_b200.so (include/unconfined_b200.h).
!
! This is the binding a maintainer of klkuhlm/unconfined adds to call the B200 library
! from the unchanged-format Fortran driver: the loop nest driver.f90:100-231 is replaced
! by ONE call to unc_eval_grid (see fortran/driver_b200.f90 and INTEGRATION.md).
! It follows the precedent of the reference's own bind(c) interface to arb_J/arb_Y
! (laplace_hankel_solutions.f90:310-325).
!
! NOTE: no Fortran compiler exists in the build image, so this file is syntax-reviewed
! only; the C side is exercised through ctypes with exactly these argument lists.
module unconfined_b200
  use, intrinsic :: iso_c_binding
  implicit none
  private
  public :: unc_params, unc_eval_grid, unc_eval_grid_ex, unc_eval_points, unc_eval_points_ex, &
       & unc_eval_screens, unc_eval_points_dz, &
       & unc_j0_zeros, unc_split_index, unc_zlay, unc_device_count, unc_set_device, &
       & unc_device_info, unc_measure_fp64_peak, unc_kernel_launch_count, unc_shutdown, &
       & unc_set_carry, unc_last_error, unc_fill_params

  integer(c_int), parameter, public :: UNC_OK = 0, UNC_ERR_BAD_ARG = -1, UNC_ERR_UNSUPPORTED = -2, &
       & UNC_ERR_NO_DEVICE = -3, UNC_ERR_CUDA = -4, UNC_ERR_IO = -5
  integer(c_int), parameter, public :: UNC_FLAG_STALE_INFINT = 1

  ! struct unc_params: field order and types as in the C header
  type, bind(C) :: unc_params
     integer(c_int32_t) :: model, M
     real(c_double)     :: alpha, tol, tee_mult
     integer(c_int32_t) :: time_type, n_time_par
     type(c_ptr)        :: time_par
     integer(c_int32_t) :: ts_k, ts_R, gl_nacc, gl_ord, n_j0z, moench_M
     type(c_ptr)        :: j0z, moench_gamma
     real(c_double)     :: kappa, alphaD, beta
     real(c_double)     :: lD, dD, bD, rDw
     real(c_double)     :: l, d, Ss, rDwobs, sF
     integer(c_int32_t) :: mn_type, mn_reserved
     real(c_double)     :: mn_ak, mn_psia, mn_psik, mn_b, mn_Sy
  end type unc_params

  interface
     integer(c_int) function unc_eval_grid(prm, nt, tD, sv, nr, rD, nz, zD, zLay, ts_scale, ngpu, &
          & totint, totintd) bind(C, name='unc_eval_grid')
       import :: c_int, c_int32_t, c_double, c_ptr, unc_params
       type(unc_params), intent(in) :: prm
       integer(c_int32_t), value :: nt, nr, nz, ngpu
       real(c_double), intent(in) :: tD(*), rD(*), zD(*)
       integer(c_int32_t), intent(in) :: sv(*), zLay(*)
       type(c_ptr), value :: ts_scale              ! c_null_ptr = fresh abscissae; else (nr,nt) doubles
       real(c_double), intent(out) :: totint(*), totintd(*)   ! (nz,nr,nt) column-major
     end function unc_eval_grid

     integer(c_int) function unc_eval_grid_ex(prm, nt, tD, sv, nr, rD, nz, zD, zLay, ts_scale, ngpu, &
          & totint, totintd, flags) bind(C, name='unc_eval_grid_ex')
       import :: c_int, c_int32_t, c_double, c_ptr, unc_params
       type(unc_params), intent(in) :: prm
       integer(c_int32_t), value :: nt, nr, nz, ngpu
       real(c_double), intent(in) :: tD(*), rD(*), zD(*)
       integer(c_int32_t), intent(in) :: sv(*), zLay(*)
       type(c_ptr), value :: ts_scale
       real(c_double), intent(out) :: totint(*), totintd(*)
       type(c_ptr), value :: flags                 ! (nz,nr,nt) int32 or c_null_ptr
     end function unc_eval_grid_ex

     integer(c_int) function unc_eval_points(prm, n, tD, sv, rD, zD, zLay, ts_scale, ngpu, s, ds) &
          & bind(C, name='unc_eval_points')
       import :: c_int, c_int32_t, c_int64_t, c_double, c_ptr, unc_params
       type(unc_params), intent(in) :: prm
       integer(c_int64_t), value :: n
       real(c_double), intent(in) :: tD(*), rD(*), zD(*)
       integer(c_int32_t), intent(in) :: sv(*), zLay(*)
       type(c_ptr), value :: ts_scale
       integer(c_int32_t), value :: ngpu
       real(c_double), intent(out) :: s(*), ds(*)
     end function unc_eval_points

     integer(c_int) function unc_eval_points_ex(prm, n, tD, sv, rD, zD, zLay, ts_scale, ngpu, s, ds, &
          & flags) bind(C, name='unc_eval_points_ex')
       import :: c_int, c_int32_t, c_int64_t, c_double, c_ptr, unc_params
       type(unc_params), intent(in) :: prm
       integer(c_int64_t), value :: n
       real(c_double), intent(in) :: tD(*), rD(*), zD(*)
       integer(c_int32_t), intent(in) :: sv(*), zLay(*)
       type(c_ptr), value :: ts_scale
       integer(c_int32_t), value :: ngpu
       real(c_double), intent(out) :: s(*), ds(*)
       type(c_ptr), value :: flags
     end function unc_eval_points_ex

     ! exact drawdown averaged over n screens [zbot, ztop] (dimensionless, 0 <= zbot < ztop <= 1);
     ! definition in include/unconfined_b200.h.  Not compiled here (no Fortran compiler in the
     ! build image); the argument list is the one tests/ exercise through ctypes.
     integer(c_int) function unc_eval_screens(prm, n, tD, sv, rD, zbot, ztop, ts_scale, ngpu, s, ds, &
          & flags) bind(C, name='unc_eval_screens')
       import :: c_int, c_int32_t, c_int64_t, c_double, c_ptr, unc_params
       type(unc_params), intent(in) :: prm
       integer(c_int64_t), value :: n
       real(c_double), intent(in) :: tD(*), rD(*), zbot(*), ztop(*)
       integer(c_int32_t), intent(in) :: sv(*)
       type(c_ptr), value :: ts_scale              ! (n) doubles or c_null_ptr
       integer(c_int32_t), value :: ngpu
       real(c_double), intent(out) :: s(*), ds(*)
       type(c_ptr), value :: flags                 ! (n) int32 or c_null_ptr
     end function unc_eval_screens

     ! vertical drawdown gradient gz = ds_D/dz_D and dgz = d gz/d ln tD at n points (dimensionless,
     ! 0 <= zD <= 1, layers geometric, no zLay); definition in include/unconfined_b200.h.  Not compiled
     ! here (no Fortran compiler in the build image); the argument list is the one tests/ exercise
     ! through ctypes.
     integer(c_int) function unc_eval_points_dz(prm, n, tD, sv, rD, zD, ts_scale, ngpu, gz, dgz, &
          & flags) bind(C, name='unc_eval_points_dz')
       import :: c_int, c_int32_t, c_int64_t, c_double, c_ptr, unc_params
       type(unc_params), intent(in) :: prm
       integer(c_int64_t), value :: n
       real(c_double), intent(in) :: tD(*), rD(*), zD(*)
       integer(c_int32_t), intent(in) :: sv(*)
       type(c_ptr), value :: ts_scale              ! (n) doubles or c_null_ptr
       integer(c_int32_t), value :: ngpu
       real(c_double), intent(out) :: gz(*), dgz(*)
       type(c_ptr), value :: flags                 ! (n) int32 or c_null_ptr
     end function unc_eval_points_dz

     integer(c_int) function unc_j0_zeros(terms, j0z) bind(C, name='unc_j0_zeros')
       import :: c_int, c_int32_t, c_double
       integer(c_int32_t), value :: terms
       real(c_double), intent(out) :: j0z(*)
     end function unc_j0_zeros

     integer(c_int) function unc_split_index(nt, tD, j0s_a, j0s_b, sv) bind(C, name='unc_split_index')
       import :: c_int, c_int32_t, c_double
       integer(c_int32_t), value :: nt, j0s_a, j0s_b
       real(c_double), intent(in) :: tD(*)
       integer(c_int32_t), intent(out) :: sv(*)
     end function unc_split_index

     integer(c_int) function unc_zlay(nz, zD, lD, dD, zLay) bind(C, name='unc_zlay')
       import :: c_int, c_int32_t, c_double
       integer(c_int32_t), value :: nz
       real(c_double), intent(in) :: zD(*)
       real(c_double), value :: lD, dD
       integer(c_int32_t), intent(out) :: zLay(*)
     end function unc_zlay

     integer(c_int) function unc_device_count(ngpu) bind(C, name='unc_device_count')
       import :: c_int, c_int32_t
       integer(c_int32_t), intent(out) :: ngpu
     end function unc_device_count

     integer(c_int) function unc_set_device(device) bind(C, name='unc_set_device')
       import :: c_int, c_int32_t
       integer(c_int32_t), value :: device
     end function unc_set_device

     integer(c_int) function unc_device_info(ngpu, fp64_peak_flops) bind(C, name='unc_device_info')
       import :: c_int, c_int32_t, c_double
       integer(c_int32_t), intent(out) :: ngpu
       real(c_double), intent(out) :: fp64_peak_flops
     end function unc_device_info

     integer(c_int) function unc_measure_fp64_peak(flops) bind(C, name='unc_measure_fp64_peak')
       import :: c_int, c_double
       real(c_double), intent(out) :: flops
     end function unc_measure_fp64_peak

     integer(c_int) function unc_kernel_launch_count(n) bind(C, name='unc_kernel_launch_count')
       import :: c_int, c_int64_t
       integer(c_int64_t), intent(out) :: n
     end function unc_kernel_launch_count

     integer(c_int) function unc_shutdown() bind(C, name='unc_shutdown')
       import :: c_int
     end function unc_shutdown

     ! default 1: grid calls that pass ts_scale also reproduce the reference's stale infint
     ! (driver.f90:205-214); 0: such points get infint = 0 (and the flag) only
     integer(c_int) function unc_set_carry(on) bind(C, name='unc_set_carry')
       import :: c_int, c_int32_t
       integer(c_int32_t), value :: on
     end function unc_set_carry

     type(c_ptr) function unc_last_error_c() bind(C, name='unc_last_error')
       import :: c_ptr
     end function unc_last_error_c
  end interface

contains

  ! Fill unc_params from the reference's own derived types (types.f90) after read_input.
  ! The arrays must be contiguous and have the TARGET attribute in the caller.
  subroutine unc_fill_params(prm, w, f, s, l, h, gl, ts, tee_mult)
    use types, only : well, formation, solution, invLaplace, invHankel, GaussLobatto, TanhSinh
    type(unc_params), intent(out) :: prm
    type(well), intent(in) :: w
    type(formation), intent(in), target :: f
    type(solution), intent(in) :: s
    type(invLaplace), intent(in), target :: l
    type(invHankel), intent(in), target :: h
    type(GaussLobatto), intent(in) :: gl
    type(TanhSinh), intent(in) :: ts
    real(c_double), intent(in) :: tee_mult
    prm%model = s%model;  prm%M = l%M
    prm%alpha = l%alpha;  prm%tol = l%tol;  prm%tee_mult = tee_mult
    prm%time_type = l%timeType
    prm%n_time_par = size(l%timePar);  prm%time_par = c_loc(l%timePar(1))
    prm%ts_k = ts%k;  prm%ts_R = ts%R
    prm%gl_nacc = gl%nacc;  prm%gl_ord = gl%ord
    prm%n_j0z = size(h%j0z);  prm%j0z = c_loc(h%j0z(1))
    prm%moench_M = f%MoenchM
    if (f%MoenchM > 0) then
       prm%moench_gamma = c_loc(f%MoenchGamma(1))
    else
       prm%moench_gamma = c_null_ptr
    end if
    prm%kappa = f%kappa;  prm%alphaD = f%alphaD;  prm%beta = f%beta
    prm%lD = w%lD;  prm%dD = w%dD;  prm%bD = w%bD;  prm%rDw = w%rDw
    prm%l = w%l;  prm%d = w%d;  prm%Ss = f%Ss;  prm%rDwobs = s%rDwobs;  prm%sF = s%sF
    ! model 6 / MNtype 1 (laplace_hankel_solutions.f90:404-442)
    prm%mn_type = s%MNtype;  prm%mn_reserved = 0
    prm%mn_ak = f%ak;  prm%mn_psia = f%psia;  prm%mn_psik = f%psik;  prm%mn_b = f%b;  prm%mn_Sy = f%Sy
  end subroutine unc_fill_params

  function unc_last_error() result(msg)
    character(len=:), allocatable :: msg
    character(kind=c_char), pointer :: p(:)
    type(c_ptr) :: cp
    integer :: n
    cp = unc_last_error_c()
    msg = ''
    if (.not. c_associated(cp)) return
    call c_f_pointer(cp, p, [512])
    n = 0
    do while (n < 512)
       if (p(n+1) == c_null_char) exit
       n = n + 1
    end do
    allocate(character(len=n) :: msg)
    msg = transfer(p(1:n), msg)
  end function unc_last_error

end module unconfined_b200
