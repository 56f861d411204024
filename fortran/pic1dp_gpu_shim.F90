! fortran/pic1dp_gpu_shim.F90 -- ISO_C_BINDING side of the drop-in boundary (include/pic1dp_gpu.h).
!
! Status: SOURCE ONLY.  No Fortran compiler, MPI or PETSc exists in the build image or on the GPU boxes, so this
! file has never been compiled; it is the binding a maintainer of PIC1D-PETSc adds (INTEGRATION.md walks through
! it).  The same call sequence is exercised against the real library from C (host/pic1dp_host.cpp) and from Python
! (pic1dp_b200/host.py, tests/).
!
! How it plugs in: the three hot-path modules keep their public procedure names and argument lists
! (src/pic1dp_particle.F90:66,145,275,819; src/pic1dp_field.F90:55,218,315; src/pic1dp_interaction.F90:33,161).
! Their bodies are replaced by the `gpu_*` procedures below, which forward to the C ABI and store the return code
! in global_ierr followed by CHKERRQ -- the reference's own error convention (src/pic1dp_global.F90:59).
! Marker Vecs stay allocated on the host (particle_load and pic1dp_output still use them); they are stale
! between gpu_particle_refresh_host calls, which the driver makes before output_all / particle_optimize.
module pic1dp_gpu
use, intrinsic :: iso_c_binding
implicit none
private

integer(c_int), parameter, public :: PIC1DP_MAX_SPECIES = 4, PIC1DP_MAX_MODES = 64
integer(c_int), parameter, public :: PIC1DP_ABI_VERSION = 2

! mirrors struct pic1dp_params (include/pic1dp_gpu.h); field order and types must match exactly
type, bind(c), public :: pic1dp_params
  integer(c_int32_t) :: abi_version
  integer(c_int32_t) :: struct_bytes
  integer(c_int32_t) :: nx
  integer(c_int32_t) :: nmode
  integer(c_int32_t) :: modes(PIC1DP_MAX_MODES)
  real(c_double) :: lx
  real(c_double) :: dt
  integer(c_int32_t) :: nspecies
  real(c_double) :: charge(PIC1DP_MAX_SPECIES)
  real(c_double) :: mass(PIC1DP_MAX_SPECIES)
  real(c_double) :: temperature(PIC1DP_MAX_SPECIES)
  real(c_double) :: temperature2(PIC1DP_MAX_SPECIES)
  real(c_double) :: density(PIC1DP_MAX_SPECIES)
  real(c_double) :: v0(PIC1DP_MAX_SPECIES)
  integer(c_int32_t) :: iptcldist
  integer(c_int32_t) :: deltaf
  integer(c_int32_t) :: linear
  integer(c_int32_t) :: iptclshape
  integer(c_int64_t) :: capacity
  integer(c_int32_t) :: device
  integer(c_int32_t) :: rank
  integer(c_int32_t) :: nranks
  integer(c_int32_t) :: deposit_mode
  integer(c_int32_t) :: field_mode
  integer(c_int32_t) :: fuse
  integer(c_int32_t) :: load_path
  integer(c_int32_t) :: arith_mode
  integer(c_int32_t) :: no_step_graph
  integer(c_int32_t) :: reserved(5)
end type pic1dp_params

interface
  subroutine pic1dp_gpu_params_default(p) bind(c, name = 'pic1dp_gpu_params_default')
    import :: pic1dp_params
    type(pic1dp_params), intent(out) :: p
  end subroutine
  integer(c_int) function pic1dp_gpu_create(p, handle) bind(c, name = 'pic1dp_gpu_create')
    import :: pic1dp_params, c_ptr, c_int
    type(pic1dp_params), intent(in) :: p
    type(c_ptr), intent(out) :: handle
  end function
  integer(c_int) function pic1dp_gpu_destroy(handle) bind(c, name = 'pic1dp_gpu_destroy')
    import :: c_ptr, c_int
    type(c_ptr), value :: handle
  end function
  integer(c_int) function pic1dp_gpu_comm_unique_id(id) bind(c, name = 'pic1dp_gpu_comm_unique_id')
    import :: c_int8_t, c_int
    integer(c_int8_t), intent(out) :: id(128)
  end function
  integer(c_int) function pic1dp_gpu_comm_init(handle, id) bind(c, name = 'pic1dp_gpu_comm_init')
    import :: c_ptr, c_int8_t, c_int
    type(c_ptr), value :: handle
    integer(c_int8_t), intent(in) :: id(128)
  end function
  integer(c_int) function pic1dp_gpu_set_markers(handle, isp, np, x, v, p, w) bind(c, name = 'pic1dp_gpu_set_markers')
    import :: c_ptr, c_int, c_int32_t, c_int64_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: isp
    integer(c_int64_t), value :: np
    real(c_double), intent(in) :: x(*), v(*), p(*), w(*)
  end function
  integer(c_int) function pic1dp_gpu_load_markers(handle, isp, np, nparticle_init, rand_v, rand_x, v_max, init_nmode, &
      init_mode, init_mode_cos, init_mode_sin) bind(c, name = 'pic1dp_gpu_load_markers')
    import :: c_ptr, c_int, c_int32_t, c_int64_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: isp, init_nmode
    integer(c_int64_t), value :: np, nparticle_init
    real(c_double), intent(in) :: rand_v(*), rand_x(*), init_mode_cos(*), init_mode_sin(*)
    real(c_double), value :: v_max
    integer(c_int32_t), intent(in) :: init_mode(*)
  end function
  integer(c_int) function pic1dp_gpu_load_markers_maxwellian(handle, isp, np, nparticle_init, gauss_v, rand_x, &
      init_nmode, init_mode, init_mode_cos, init_mode_sin) bind(c, name = 'pic1dp_gpu_load_markers_maxwellian')
    import :: c_ptr, c_int, c_int32_t, c_int64_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: isp, init_nmode
    integer(c_int64_t), value :: np, nparticle_init
    real(c_double), intent(in) :: gauss_v(*), rand_x(*), init_mode_cos(*), init_mode_sin(*)
    integer(c_int32_t), intent(in) :: init_mode(*)
  end function
  integer(c_int) function pic1dp_gpu_load_markers_kiss64(handle, isp, np, nparticle_init, seeds, offset_v, offset_x, &
      v_max, init_nmode, init_mode, init_mode_cos, init_mode_sin) bind(c, name = 'pic1dp_gpu_load_markers_kiss64')
    import :: c_ptr, c_int, c_int32_t, c_int64_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: isp, init_nmode
    integer(c_int64_t), value :: np, nparticle_init, offset_v, offset_x
    integer(c_int64_t), intent(in) :: seeds(4)   ! multirand_seeds(0:3), same bits as the C uint64_t
    real(c_double), value :: v_max
    real(c_double), intent(in) :: init_mode_cos(*), init_mode_sin(*)
    integer(c_int32_t), intent(in) :: init_mode(*)
  end function
  integer(c_int) function pic1dp_host_kiss64_jump(seeds, n) bind(c, name = 'pic1dp_host_kiss64_jump')
    import :: c_int, c_int64_t
    integer(c_int64_t), intent(inout) :: seeds(4)
    integer(c_int64_t), value :: n
  end function
  integer(c_int) function pic1dp_gpu_load_markers_superkiss64(handle, isp, np, nlocal, nparticle_init, seeds, iseed, &
      v_max, init_nmode, init_mode, init_mode_cos, init_mode_sin) bind(c, name = 'pic1dp_gpu_load_markers_superkiss64')
    import :: c_ptr, c_int, c_int32_t, c_int64_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: isp, init_nmode
    integer(c_int64_t), value :: np, nlocal, nparticle_init
    integer(c_int64_t), intent(inout) :: seeds(20635)   ! multirand_seeds(0:20634), same bits as the C uint64_t
    integer(c_int32_t), intent(inout) :: iseed
    real(c_double), value :: v_max
    real(c_double), intent(in) :: init_mode_cos(*), init_mode_sin(*)
    integer(c_int32_t), intent(in) :: init_mode(*)
  end function
  integer(c_int) function pic1dp_gpu_load_markers_maxwellian_kiss64(handle, isp, np, nlocal, nparticle_init, seeds, &
      gauss_filled, gauss_buf, init_nmode, init_mode, init_mode_cos, init_mode_sin) &
      bind(c, name = 'pic1dp_gpu_load_markers_maxwellian_kiss64')
    import :: c_ptr, c_int, c_int32_t, c_int64_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: isp, init_nmode
    integer(c_int64_t), value :: np, nlocal, nparticle_init
    integer(c_int64_t), intent(inout) :: seeds(4)   ! multirand_seeds(0:3), same bits as the C uint64_t
    integer(c_int32_t), intent(inout) :: gauss_filled
    real(c_double), intent(inout) :: gauss_buf
    real(c_double), intent(in) :: init_mode_cos(*), init_mode_sin(*)
    integer(c_int32_t), intent(in) :: init_mode(*)
  end function
  integer(c_int) function pic1dp_gpu_load_markers_maxwellian_superkiss64(handle, isp, np, nlocal, nparticle_init, &
      seeds, iseed, gauss_filled, gauss_buf, init_nmode, init_mode, init_mode_cos, init_mode_sin) &
      bind(c, name = 'pic1dp_gpu_load_markers_maxwellian_superkiss64')
    import :: c_ptr, c_int, c_int32_t, c_int64_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: isp, init_nmode
    integer(c_int64_t), value :: np, nlocal, nparticle_init
    integer(c_int64_t), intent(inout) :: seeds(20635)   ! multirand_seeds(0:20634), same bits as the C uint64_t
    integer(c_int32_t), intent(inout) :: iseed, gauss_filled
    real(c_double), intent(inout) :: gauss_buf
    real(c_double), intent(in) :: init_mode_cos(*), init_mode_sin(*)
    integer(c_int32_t), intent(in) :: init_mode(*)
  end function
  integer(c_int) function pic1dp_gpu_output_all(handle, nx_opd, nv_opd, v_max, scalars, dist) &
      bind(c, name = 'pic1dp_gpu_output_all')
    import :: c_ptr, c_int, c_int32_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: nx_opd, nv_opd
    real(c_double), value :: v_max
    real(c_double), intent(out) :: scalars(*), dist(*)
  end function
  integer(c_int) function pic1dp_gpu_get_markers(handle, isp, x, v, p, w, np) bind(c, name = 'pic1dp_gpu_get_markers')
    import :: c_ptr, c_int, c_int32_t, c_int64_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: isp
    real(c_double), intent(out) :: x(*), v(*), p(*), w(*)
    integer(c_int64_t), intent(out) :: np
  end function
  integer(c_int) function pic1dp_gpu_compute_shape_x(handle) bind(c, name = 'pic1dp_gpu_compute_shape_x')
    import :: c_ptr, c_int
    type(c_ptr), value :: handle
  end function
  integer(c_int) function pic1dp_gpu_collect_charge(handle) bind(c, name = 'pic1dp_gpu_collect_charge')
    import :: c_ptr, c_int
    type(c_ptr), value :: handle
  end function
  integer(c_int) function pic1dp_gpu_solve_field(handle) bind(c, name = 'pic1dp_gpu_solve_field')
    import :: c_ptr, c_int
    type(c_ptr), value :: handle
  end function
  integer(c_int) function pic1dp_gpu_push(handle, irk) bind(c, name = 'pic1dp_gpu_push')
    import :: c_ptr, c_int, c_int32_t
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: irk
  end function
  integer(c_int) function pic1dp_gpu_get_field(handle, electric, chargeden, mode_re, mode_im) &
      bind(c, name = 'pic1dp_gpu_get_field')
    import :: c_ptr, c_int, c_double
    type(c_ptr), value :: handle
    real(c_double), intent(out) :: electric(*), chargeden(*), mode_re(*), mode_im(*)
  end function
  integer(c_int) function pic1dp_gpu_set_field(handle, electric, chargeden) bind(c, name = 'pic1dp_gpu_set_field')
    import :: c_ptr, c_int
    type(c_ptr), value :: handle
    type(c_ptr), value :: electric, chargeden   ! const double*, either may be c_null_ptr
  end function
  integer(c_int) function pic1dp_gpu_p2p_export(handle, ipc) bind(c, name = 'pic1dp_gpu_p2p_export')
    import :: c_ptr, c_int8_t, c_int
    type(c_ptr), value :: handle
    integer(c_int8_t), intent(out) :: ipc(64)
  end function
  integer(c_int) function pic1dp_gpu_p2p_import(handle, all_ipc) bind(c, name = 'pic1dp_gpu_p2p_import')
    import :: c_ptr, c_int8_t, c_int
    type(c_ptr), value :: handle
    integer(c_int8_t), intent(in) :: all_ipc(*)
  end function
  integer(c_int) function pic1dp_gpu_output_field(handle, scalars) bind(c, name = 'pic1dp_gpu_output_field')
    import :: c_ptr, c_int, c_double
    type(c_ptr), value :: handle
    real(c_double), intent(out) :: scalars(*)
  end function
  integer(c_int) function pic1dp_gpu_output_ptcldist(handle, isp, nx_opd, nv_opd, v_max, markr_xv, total_xv, &
      pertb_xv, markr_v, total_v, pertb_v) bind(c, name = 'pic1dp_gpu_output_ptcldist')
    import :: c_ptr, c_int, c_int32_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: isp, nx_opd, nv_opd
    real(c_double), value :: v_max
    real(c_double), intent(out) :: markr_xv(*), total_xv(*), pertb_xv(*), markr_v(*), total_v(*), pertb_v(*)
  end function
  integer(c_int) function pic1dp_gpu_sync(handle) bind(c, name = 'pic1dp_gpu_sync')
    import :: c_ptr, c_int
    type(c_ptr), value :: handle
  end function
  ! marker optimisation (src/pic1dp_particle.F90:356-746)
  integer(c_int) function pic1dp_gpu_compute_dist_pertb_abs_v(handle, nv, v_max, dist) &
      bind(c, name = 'pic1dp_gpu_compute_dist_pertb_abs_v')
    import :: c_ptr, c_int, c_int32_t, c_double
    type(c_ptr), value :: handle
    integer(c_int32_t), value :: nv
    real(c_double), value :: v_max
    real(c_double), intent(out) :: dist(*)   ! [nv, nspecies] in Fortran order
  end function
  integer(c_int) function pic1dp_gpu_particle_merge(handle, thsh, np_out) bind(c, name = 'pic1dp_gpu_particle_merge')
    import :: c_ptr, c_int, c_int64_t, c_double
    type(c_ptr), value :: handle
    real(c_double), value :: thsh
    integer(c_int64_t), intent(out) :: np_out(*)
  end function
  integer(c_int) function pic1dp_gpu_particle_remove(handle, thsh, typeremove, remove_frac, dice, rng_ctx, np_out) &
      bind(c, name = 'pic1dp_gpu_particle_remove')
    import :: c_ptr, c_funptr, c_int, c_int32_t, c_int64_t, c_double
    type(c_ptr), value :: handle
    real(c_double), value :: thsh, remove_frac
    integer(c_int32_t), value :: typeremove
    type(c_funptr), value :: dice
    type(c_ptr), value :: rng_ctx
    integer(c_int64_t), intent(out) :: np_out(*)
  end function
  integer(c_int) function pic1dp_gpu_particle_split(handle, thsh, ngroup, dv_sig_frac, gauss, rng_ctx, np_out) &
      bind(c, name = 'pic1dp_gpu_particle_split')
    import :: c_ptr, c_funptr, c_int, c_int32_t, c_int64_t, c_double
    type(c_ptr), value :: handle
    real(c_double), value :: thsh, dv_sig_frac
    integer(c_int32_t), value :: ngroup
    type(c_funptr), value :: gauss
    type(c_ptr), value :: rng_ctx
    integer(c_int64_t), intent(out) :: np_out(*)
  end function
end interface

type(c_ptr), save, public :: gpu_handle = c_null_ptr

public :: pic1dp_gpu_params_default, pic1dp_gpu_create, pic1dp_gpu_destroy
public :: pic1dp_gpu_comm_unique_id, pic1dp_gpu_comm_init
public :: pic1dp_gpu_set_markers, pic1dp_gpu_load_markers, pic1dp_gpu_load_markers_maxwellian
public :: pic1dp_gpu_get_markers, pic1dp_gpu_compute_shape_x
public :: pic1dp_gpu_collect_charge, pic1dp_gpu_solve_field, pic1dp_gpu_push
public :: pic1dp_gpu_get_field, pic1dp_gpu_set_field, pic1dp_gpu_sync
public :: pic1dp_gpu_p2p_export, pic1dp_gpu_p2p_import, pic1dp_gpu_output_field, pic1dp_gpu_output_ptcldist
public :: pic1dp_gpu_compute_dist_pertb_abs_v, pic1dp_gpu_particle_merge, pic1dp_gpu_particle_remove
public :: pic1dp_gpu_particle_split
public :: pic1dp_gpu_load_markers_kiss64, pic1dp_host_kiss64_jump, pic1dp_gpu_output_all
public :: pic1dp_gpu_load_markers_superkiss64
public :: pic1dp_gpu_load_markers_maxwellian_kiss64, pic1dp_gpu_load_markers_maxwellian_superkiss64

end module pic1dp_gpu


! ----------------------------------------------------------------------------------------------------------------
! Replacement bodies.  Each `gpu_*` subroutine below is what the reference procedure of the same role calls (or
! becomes) when the code is built with -D__PIC1DP_GPU.  They live in one module here for readability; in the
! reference tree they go into pic1dp_particle / pic1dp_field / pic1dp_interaction (see INTEGRATION.md).
! ----------------------------------------------------------------------------------------------------------------
module pic1dp_gpu_glue
use, intrinsic :: iso_c_binding
use pic1dp_gpu
use pic1dp_global   ! global_ierr, global_irk, global_mype, global_npe
use pic1dp_input    ! input_* parameters
implicit none
#include "finclude/petscdef.h"

contains

! particle_init + field_init: after the reference has created its host Vecs (src/pic1dp_particle.F90:89-129,
! src/pic1dp_field.F90:67-155), create the device-resident state.
subroutine gpu_init(local_capacity)
implicit none
#include "finclude/petsc.h90"
PetscInt, intent(in) :: local_capacity   ! particle_ip_high - particle_ip_low
type(pic1dp_params) :: p
integer(c_int8_t) :: id(128), ipc_mine(64), ipc_all(64 * 8)
integer :: imode

call pic1dp_gpu_params_default(p)
p%nx = input_nx
p%nmode = input_nmode
do imode = 0, input_nmode - 1
  p%modes(imode + 1) = input_modes(imode)
end do
p%lx = input_lx
p%dt = input_dt
p%nspecies = input_nspecies
p%charge(1 : input_nspecies) = input_species_charge
p%mass(1 : input_nspecies) = input_species_mass
p%temperature(1 : input_nspecies) = input_species_temperature
p%temperature2(1 : input_nspecies) = input_species_temperature2
p%density(1 : input_nspecies) = input_species_density
p%v0(1 : input_nspecies) = input_species_v0
p%iptcldist = input_iptcldist
p%deltaf = input_deltaf
p%linear = input_linear
p%iptclshape = input_iptclshape
p%capacity = local_capacity
p%device = mod(global_mype, 8)      ! one MPI rank per GPU of the box
p%rank = global_mype
p%nranks = global_npe

global_ierr = pic1dp_gpu_create(p, gpu_handle)
CHKERRQ(global_ierr)

if (global_npe > 1) then
  ! replaces MPI_COMM_WORLD for the density all-reduce (src/pic1dp_interaction.F90:132-133)
  if (global_mype == 0) then
    global_ierr = pic1dp_gpu_comm_unique_id(id)
    CHKERRQ(global_ierr)
  end if
  call MPI_Bcast(id, 128, MPI_BYTE, 0, MPI_COMM_WORLD, global_ierr)
  CHKERRQ(global_ierr)
  global_ierr = pic1dp_gpu_comm_init(gpu_handle, id)
  CHKERRQ(global_ierr)
  ! optional: density all-reduce through peer memory (NVLink) instead of ncclAllReduce
  if (global_npe <= 8) then
    global_ierr = pic1dp_gpu_p2p_export(gpu_handle, ipc_mine)
    CHKERRQ(global_ierr)
    call MPI_Allgather(ipc_mine, 64, MPI_BYTE, ipc_all, 64, MPI_BYTE, MPI_COMM_WORLD, global_ierr)
    CHKERRQ(global_ierr)
    global_ierr = pic1dp_gpu_p2p_import(gpu_handle, ipc_all)
    CHKERRQ(global_ierr)
  end if
end if
end subroutine gpu_init

! after particle_load (src/pic1dp_particle.F90:145-269): host Vecs -> device
subroutine gpu_particle_upload(ispecies, np, vx, vv, vp, vw)
implicit none
#include "finclude/petsc.h90"
PetscInt, intent(in) :: ispecies, np
Vec, intent(in) :: vx, vv, vp, vw
PetscScalar, dimension(:), pointer :: px, pv, pp, pw

call VecGetArrayF90(vx, px, global_ierr)
CHKERRQ(global_ierr)
call VecGetArrayF90(vv, pv, global_ierr)
CHKERRQ(global_ierr)
call VecGetArrayF90(vp, pp, global_ierr)
CHKERRQ(global_ierr)
call VecGetArrayF90(vw, pw, global_ierr)
CHKERRQ(global_ierr)
global_ierr = pic1dp_gpu_set_markers(gpu_handle, int(ispecies - 1, c_int32_t), int(np, c_int64_t), px, pv, pp, pw)
CHKERRQ(global_ierr)
call VecRestoreArrayF90(vx, px, global_ierr)
CHKERRQ(global_ierr)
call VecRestoreArrayF90(vv, pv, global_ierr)
CHKERRQ(global_ierr)
call VecRestoreArrayF90(vp, pp, global_ierr)
CHKERRQ(global_ierr)
call VecRestoreArrayF90(vw, pw, global_ierr)
CHKERRQ(global_ierr)
end subroutine gpu_particle_upload

! alternative to gpu_particle_upload: particle_load keeps only its two multirand_real_array calls
! (src/pic1dp_particle.F90:180, :222) and hands the raw uniform streams over; the loader arithmetic (:181-237,
! :260-263) runs on the device, so 16 instead of 32 bytes per marker cross PCIe
subroutine gpu_particle_load(ispecies, np, rand_v, rand_x)
implicit none
#include "finclude/petsc.h90"
PetscInt, intent(in) :: ispecies, np
PetscScalar, dimension(:), intent(in) :: rand_v, rand_x
global_ierr = pic1dp_gpu_load_markers(gpu_handle, int(ispecies - 1, c_int32_t), int(np, c_int64_t), &
  int(input_species_nparticle_init(ispecies), c_int64_t), rand_v, rand_x, real(input_v_max, c_double), &
  int(input_init_nmode, c_int32_t), int(input_init_mode, c_int32_t), real(input_init_mode_cos, c_double), &
  real(input_init_mode_sin, c_double))
CHKERRQ(global_ierr)
end subroutine gpu_particle_load

! particle_load with input_multirand_al_int = 1 (KISS64): no marker-sized host-to-device copy.  Call in place of the two
! multirand_real_array calls (src/pic1dp_particle.F90:180, :222) AFTER multirand_init (:159-160): the device generates
! exactly the numbers those calls would have produced, and the host generator is advanced past them so that later draws
! (particle_remove, particle_split) continue the same stream.  nlocal = particle_ip_high - particle_ip_low.
subroutine gpu_particle_load_kiss64(ispecies, np, nlocal)
use multirand, only : multirand_seeds
implicit none
#include "finclude/petsc.h90"
PetscInt, intent(in) :: ispecies, np, nlocal
integer(c_int64_t) :: seeds(4), off_v
seeds(1 : 4) = multirand_seeds(0 : 3)
off_v = 0_c_int64_t                          ! multirand_seeds already stands at this species' first draw
global_ierr = pic1dp_gpu_load_markers_kiss64(gpu_handle, int(ispecies - 1, c_int32_t), int(np, c_int64_t), &
  int(input_species_nparticle_init(ispecies), c_int64_t), seeds, off_v, off_v + int(nlocal, c_int64_t), &
  real(input_v_max, c_double), int(input_init_nmode, c_int32_t), int(input_init_mode, c_int32_t), &
  real(input_init_mode_cos, c_double), real(input_init_mode_sin, c_double))
CHKERRQ(global_ierr)
global_ierr = pic1dp_host_kiss64_jump(seeds, 2_c_int64_t * int(nlocal, c_int64_t))
CHKERRQ(global_ierr)
multirand_seeds(0 : 3) = seeds(1 : 4)
end subroutine gpu_particle_load_kiss64

! particle_load with input_multirand_al_int = 3 (SuperKISS64, the default input): no marker-sized host-to-device copy.
! Call in place of the two multirand_real_array calls (src/pic1dp_particle.F90:180, :222) AFTER multirand_init
! (:159-160).  The device generates exactly the 2 * nlocal numbers those calls would have drawn and returns the advanced
! state (table, carry, LCG, xorshift and table position), which is copied back into the multirand module so that later
! draws (particle_remove, particle_split) continue the same stream.  nlocal = particle_ip_high - particle_ip_low.
subroutine gpu_particle_load_superkiss64(ispecies, np, nlocal)
use multirand, only : multirand_seeds, multirand_iseed
implicit none
#include "finclude/petsc.h90"
PetscInt, intent(in) :: ispecies, np, nlocal
integer(c_int64_t) :: seeds(20635)
integer(c_int32_t) :: iseed
seeds(1 : 20635) = multirand_seeds(0 : 20634)
iseed = int(multirand_iseed, c_int32_t)
global_ierr = pic1dp_gpu_load_markers_superkiss64(gpu_handle, int(ispecies - 1, c_int32_t), int(np, c_int64_t), &
  int(nlocal, c_int64_t), int(input_species_nparticle_init(ispecies), c_int64_t), seeds, iseed, &
  real(input_v_max, c_double), int(input_init_nmode, c_int32_t), int(input_init_mode, c_int32_t), &
  real(input_init_mode_cos, c_double), real(input_init_mode_sin, c_double))
CHKERRQ(global_ierr)
multirand_seeds(0 : 20634) = seeds(1 : 20635)
multirand_iseed = iseed
end subroutine gpu_particle_load_superkiss64

! particle_load with input_imarker = 1 (Maxwellian markers, iptcldist = 0): no marker-sized host-to-device copy.  Call in
! place of multirand_gaussian_array(pv) and multirand_real_array(px) (src/pic1dp_particle.F90:172-178, :222) AFTER
! multirand_init.  The device draws exactly what those two calls would have drawn (src/multirand.F90:838-872, then :664)
! and returns the advanced state, which is copied back into the multirand module.  gauss_filled / gauss_buf are the
! one-slot buffer of multirand_gaussian_array (a value left over by an odd-length call): pass the module's buffer and
! store the returned one back, so that the next Gaussian draws (the next species, particle_split) continue the stream.
subroutine gpu_particle_load_maxwellian_kiss64(ispecies, np, nlocal, gauss_filled, gauss_buf)
use multirand, only : multirand_seeds
implicit none
#include "finclude/petsc.h90"
PetscInt, intent(in) :: ispecies, np, nlocal
integer(c_int32_t), intent(inout) :: gauss_filled
real(c_double), intent(inout) :: gauss_buf
integer(c_int64_t) :: seeds(4)
seeds(1 : 4) = multirand_seeds(0 : 3)
global_ierr = pic1dp_gpu_load_markers_maxwellian_kiss64(gpu_handle, int(ispecies - 1, c_int32_t), int(np, c_int64_t), &
  int(nlocal, c_int64_t), int(input_species_nparticle_init(ispecies), c_int64_t), seeds, gauss_filled, gauss_buf, &
  int(input_init_nmode, c_int32_t), int(input_init_mode, c_int32_t), &
  real(input_init_mode_cos, c_double), real(input_init_mode_sin, c_double))
CHKERRQ(global_ierr)
multirand_seeds(0 : 3) = seeds(1 : 4)
end subroutine gpu_particle_load_maxwellian_kiss64

subroutine gpu_particle_load_maxwellian_superkiss64(ispecies, np, nlocal, gauss_filled, gauss_buf)
use multirand, only : multirand_seeds, multirand_iseed
implicit none
#include "finclude/petsc.h90"
PetscInt, intent(in) :: ispecies, np, nlocal
integer(c_int32_t), intent(inout) :: gauss_filled
real(c_double), intent(inout) :: gauss_buf
integer(c_int64_t) :: seeds(20635)
integer(c_int32_t) :: iseed
seeds(1 : 20635) = multirand_seeds(0 : 20634)
iseed = int(multirand_iseed, c_int32_t)
global_ierr = pic1dp_gpu_load_markers_maxwellian_superkiss64(gpu_handle, int(ispecies - 1, c_int32_t), &
  int(np, c_int64_t), int(nlocal, c_int64_t), int(input_species_nparticle_init(ispecies), c_int64_t), seeds, iseed, &
  gauss_filled, gauss_buf, int(input_init_nmode, c_int32_t), int(input_init_mode, c_int32_t), &
  real(input_init_mode_cos, c_double), real(input_init_mode_sin, c_double))
CHKERRQ(global_ierr)
multirand_seeds(0 : 20634) = seeds(1 : 20635)
multirand_iseed = iseed
end subroutine gpu_particle_load_maxwellian_superkiss64

! before output_all / particle_optimize (src/pic1dp_output.F90:128-150, :228-237): device -> host Vecs
subroutine gpu_particle_refresh_host(ispecies, vx, vv, vp, vw)
implicit none
#include "finclude/petsc.h90"
PetscInt, intent(in) :: ispecies
Vec, intent(in) :: vx, vv, vp, vw
PetscScalar, dimension(:), pointer :: px, pv, pp, pw
integer(c_int64_t) :: np

call VecGetArrayF90(vx, px, global_ierr)
CHKERRQ(global_ierr)
call VecGetArrayF90(vv, pv, global_ierr)
CHKERRQ(global_ierr)
call VecGetArrayF90(vp, pp, global_ierr)
CHKERRQ(global_ierr)
call VecGetArrayF90(vw, pw, global_ierr)
CHKERRQ(global_ierr)
global_ierr = pic1dp_gpu_get_markers(gpu_handle, int(ispecies - 1, c_int32_t), px, pv, pp, pw, np)
CHKERRQ(global_ierr)
call VecRestoreArrayF90(vx, px, global_ierr)
CHKERRQ(global_ierr)
call VecRestoreArrayF90(vv, pv, global_ierr)
CHKERRQ(global_ierr)
call VecRestoreArrayF90(vp, pp, global_ierr)
CHKERRQ(global_ierr)
call VecRestoreArrayF90(vw, pw, global_ierr)
CHKERRQ(global_ierr)
end subroutine gpu_particle_refresh_host

! body of particle_compute_shape_x (src/pic1dp_particle.F90:275-350)
subroutine gpu_particle_compute_shape_x
implicit none
#include "finclude/petsc.h90"
global_ierr = pic1dp_gpu_compute_shape_x(gpu_handle)
CHKERRQ(global_ierr)
end subroutine gpu_particle_compute_shape_x

! body of interaction_collect_charge (src/pic1dp_interaction.F90:33-155)
subroutine gpu_interaction_collect_charge
implicit none
#include "finclude/petsc.h90"
global_ierr = pic1dp_gpu_collect_charge(gpu_handle)
CHKERRQ(global_ierr)
end subroutine gpu_interaction_collect_charge

! body of field_solve_electric (src/pic1dp_field.F90:218-270)
subroutine gpu_field_solve_electric
implicit none
#include "finclude/petsc.h90"
global_ierr = pic1dp_gpu_solve_field(gpu_handle)
CHKERRQ(global_ierr)
end subroutine gpu_field_solve_electric

! body of interaction_push_particle (src/pic1dp_interaction.F90:161-370); global_irk is the implicit input
subroutine gpu_interaction_push_particle
implicit none
#include "finclude/petsc.h90"
global_ierr = pic1dp_gpu_push(gpu_handle, int(global_irk, c_int32_t))
CHKERRQ(global_ierr)
end subroutine gpu_interaction_push_particle

! before output_field (src/pic1dp_output.F90:178-187): replicated grid quantities -> the local slices of the
! distributed field Vecs.  ebuf/rbuf are host work arrays of length input_nx, mre/mim of length input_nmode.
subroutine gpu_field_refresh_host(v_electric, v_chargeden, v_mode_re, v_mode_im, ix_low, ix_high, im_low, im_high)
implicit none
#include "finclude/petsc.h90"
Vec, intent(in) :: v_electric, v_chargeden, v_mode_re, v_mode_im
PetscInt, intent(in) :: ix_low, ix_high, im_low, im_high
real(c_double) :: ebuf(0 : input_nx - 1), rbuf(0 : input_nx - 1)
real(c_double) :: mre(0 : input_nmode - 1), mim(0 : input_nmode - 1)
PetscScalar, dimension(:), pointer :: pa

global_ierr = pic1dp_gpu_get_field(gpu_handle, ebuf, rbuf, mre, mim)
CHKERRQ(global_ierr)
call VecGetArrayF90(v_electric, pa, global_ierr)
CHKERRQ(global_ierr)
pa(1 : ix_high - ix_low) = ebuf(ix_low : ix_high - 1)
call VecRestoreArrayF90(v_electric, pa, global_ierr)
CHKERRQ(global_ierr)
call VecGetArrayF90(v_chargeden, pa, global_ierr)
CHKERRQ(global_ierr)
pa(1 : ix_high - ix_low) = rbuf(ix_low : ix_high - 1)
call VecRestoreArrayF90(v_chargeden, pa, global_ierr)
CHKERRQ(global_ierr)
if (im_high > im_low) then
  call VecGetArrayF90(v_mode_re, pa, global_ierr)
  CHKERRQ(global_ierr)
  pa(1 : im_high - im_low) = mre(im_low : im_high - 1)
  call VecRestoreArrayF90(v_mode_re, pa, global_ierr)
  CHKERRQ(global_ierr)
  call VecGetArrayF90(v_mode_im, pa, global_ierr)
  CHKERRQ(global_ierr)
  pa(1 : im_high - im_low) = mim(im_low : im_high - 1)
  call VecRestoreArrayF90(v_mode_im, pa, global_ierr)
  CHKERRQ(global_ierr)
end if
end subroutine gpu_field_refresh_host

! field_test (src/pic1dp_field.F90:276-309): the reference fills field_chargeden on the host with VecSetValues; the
! replicated device copy of rho takes the same values, then field_solve_electric runs on the device as usual
subroutine gpu_field_test_set_chargeden
implicit none
#include "finclude/petsc.h90"
real(c_double), target :: values(0 : input_nx - 1)
PetscInt :: ix
do ix = 0, input_nx - 1
  values(ix) = cos(2.0_kpr * PETSC_PI * ix / real(input_nx, kpr))
end do
global_ierr = pic1dp_gpu_set_field(gpu_handle, c_null_ptr, c_loc(values))
CHKERRQ(global_ierr)
end subroutine gpu_field_test_set_chargeden

! scalar part of output_field (src/pic1dp_output.F90:117-172) from device-side reductions: realbuf(2:) of the
! reference = scalars(1:1+3*nspecies); no marker array crosses PCIe
subroutine gpu_output_field_scalars(realbuf)
implicit none
#include "finclude/petsc.h90"
PetscReal, dimension(2 + input_nspecies * 3), intent(inout) :: realbuf
real(c_double) :: scalars(1 + 3 * input_nspecies)
global_ierr = pic1dp_gpu_output_field(gpu_handle, scalars)
CHKERRQ(global_ierr)
realbuf(2 : 2 + 3 * input_nspecies) = scalars(1 : 1 + 3 * input_nspecies)
end subroutine gpu_output_field_scalars

! the six arrays of output_ptcldist (src/pic1dp_output.F90:196-477) for one species, binned on the device
subroutine gpu_output_ptcldist(ispecies, markr_xv, total_xv, pertb_xv, markr_v, total_v, pertb_v)
implicit none
#include "finclude/petsc.h90"
PetscInt, intent(in) :: ispecies
PetscScalar, dimension(0 : input_nx_opd * input_nv_opd - 1), intent(out) :: markr_xv, total_xv, pertb_xv
PetscScalar, dimension(0 : input_nv_opd - 1), intent(out) :: markr_v, total_v, pertb_v
global_ierr = pic1dp_gpu_output_ptcldist(gpu_handle, int(ispecies - 1, c_int32_t), int(input_nx_opd, c_int32_t), &
  int(input_nv_opd, c_int32_t), real(input_v_max, c_double), markr_xv, total_xv, pertb_xv, markr_v, total_v, pertb_v)
CHKERRQ(global_ierr)
end subroutine gpu_output_ptcldist

! ---- marker optimisation: bodies of particle_compute_dist_pertb_abs_v / particle_merge / particle_remove /
! particle_split (src/pic1dp_particle.F90:356-746).  particle_optimize (:752-813) itself is unchanged: it still
! decides WHEN, these decide HOW.  The RNG stays the host's multirand module; the library draws from it through two
! bind(C) call-backs so that the stream is consumed in the reference's visiting order.
function gpu_cb_real64(ctx) bind(c) result(r)
use multirand
implicit none
type(c_ptr), value :: ctx
real(c_double) :: r
r = multirand_real64()
end function gpu_cb_real64

subroutine gpu_cb_gaussian_array(ctx, a, n) bind(c)
use multirand
implicit none
type(c_ptr), value :: ctx
integer(c_int32_t), value :: n
real(c_double), intent(out) :: a(n)
call multirand_gaussian_array(a)
end subroutine gpu_cb_gaussian_array

subroutine gpu_particle_compute_dist_pertb_abs_v(dist_pertb_abs_v)
implicit none
#include "finclude/petsc.h90"
PetscScalar, dimension(input_nspecies, 0 : input_nv - 1), intent(out) :: dist_pertb_abs_v
real(c_double) :: dist(0 : input_nv - 1, input_nspecies)   ! C layout [nspecies][nv]
global_ierr = pic1dp_gpu_compute_dist_pertb_abs_v(gpu_handle, int(input_nv, c_int32_t), real(input_v_max, c_double), dist)
CHKERRQ(global_ierr)
dist_pertb_abs_v = transpose(dist)
end subroutine gpu_particle_compute_dist_pertb_abs_v

subroutine gpu_particle_merge(thsh, np)
implicit none
#include "finclude/petsc.h90"
PetscReal, intent(in) :: thsh
PetscInt, dimension(input_nspecies), intent(out) :: np   ! particle_np
integer(c_int64_t) :: np64(input_nspecies)
global_ierr = pic1dp_gpu_particle_merge(gpu_handle, real(thsh, c_double), np64)
CHKERRQ(global_ierr)
np = int(np64, kind(np))
end subroutine gpu_particle_merge

subroutine gpu_particle_remove(thsh, np)
implicit none
#include "finclude/petsc.h90"
PetscReal, intent(in) :: thsh
PetscInt, dimension(input_nspecies), intent(out) :: np
integer(c_int64_t) :: np64(input_nspecies)
global_ierr = pic1dp_gpu_particle_remove(gpu_handle, real(thsh, c_double), int(input_typeremove, c_int32_t), &
  real(input_remove_frac, c_double), c_funloc(gpu_cb_real64), c_null_ptr, np64)
CHKERRQ(global_ierr)
np = int(np64, kind(np))
end subroutine gpu_particle_remove

subroutine gpu_particle_split(thsh, np)
implicit none
#include "finclude/petsc.h90"
PetscReal, intent(in) :: thsh
PetscInt, dimension(input_nspecies), intent(out) :: np
integer(c_int64_t) :: np64(input_nspecies)
global_ierr = pic1dp_gpu_particle_split(gpu_handle, real(thsh, c_double), int(input_split_ngroup, c_int32_t), &
  real(input_split_dv_sig_frac, c_double), c_funloc(gpu_cb_gaussian_array), c_null_ptr, np64)
CHKERRQ(global_ierr)
np = int(np64, kind(np))
end subroutine gpu_particle_split

! particle_final + field_final (src/pic1dp_particle.F90:819-858, src/pic1dp_field.F90:315-348)
subroutine gpu_final
implicit none
#include "finclude/petsc.h90"
global_ierr = pic1dp_gpu_destroy(gpu_handle)
CHKERRQ(global_ierr)
gpu_handle = c_null_ptr
end subroutine gpu_final

end module pic1dp_gpu_glue
