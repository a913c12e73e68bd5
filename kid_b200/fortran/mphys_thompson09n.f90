! mphys_thompson09n.f90 - drop-in replacement of KiD's interface module of the same name
! (reference: /root/reference/mphys_thompson09n.f90, "I:").  Same module name, same subroutine name
! and the same no-argument call (I:9, I:28): KiD's mphys dispatch needs no change.  The body keeps the
! host in Fortran and hands the columns to the CUDA library through iso_c_binding (include/kidmp.h):
!
!   first call : kidmp_init        replaces  call thompson_init            (I:100-103, M:374-797)
!   every call : kidmp_kid_interface replaces the gather, `call mp_thompson` per column and the
!                tendency back-out                                          (I:54-97, I:143-152, I:198-245)
!   save_dg    : unchanged, fed from the returned precipitation arrays      (I:155-192, I:248-308)
!
! NOT COMPILED IN THIS REPOSITORY'S BUILD CONTAINER (it has no Fortran compiler); the identical C ABI
! is exercised by tests/ through ctypes.  Build on a KiD machine:
!   gfortran -O3 -c mphys_thompson09n.f90   and link KiD with  -L<repo>/kid_b200 -lkidmp -lcudart
module mphys_thompson09n

  Use, intrinsic :: iso_c_binding
  Use parameters, only : num_h_moments, num_h_bins, nspecies, nz, dt &
       , h_names, mom_units, max_char_len, nx
  Use column_variables
  Use physconst, only : p0, r_on_cp, pi
  Use namelists, only : iiwarm, set_Nc
  Use switches, only : l_sediment, l_reuse_thompson_lookup
  Use diagnostics, only: save_dg, i_dgtime

  Implicit None

  ! include/kidmp.h :: kidmp_config
  type, bind(C) :: kidmp_config
     real(c_float)  :: set_Nc
     integer(c_int) :: iiwarm, l_sediment, wp_double, device, reuse_tables
     type(c_ptr)    :: table_cache_path
     integer(c_int) :: ndev                       ! > 1: one handle over ndev GPUs, columns cut into ndev ranges
     type(c_ptr)    :: device_ids                 ! ndev CUDA ordinals, c_null_ptr = 0 .. ndev-1
  end type kidmp_config

  ! include/kidmp.h :: kidmp_kid_columns
  type, bind(C) :: kidmp_kid_columns
     integer(c_long) :: nx
     integer(c_int)  :: nz
     type(c_ptr) :: theta, dtheta_adv, dtheta_div, exner, qv, dqv_adv, dqv_div, dz
     type(c_ptr) :: hyd(7), dhyd_adv(7), dhyd_div(7)
     type(c_ptr) :: dtheta_mphys, dqv_mphys, dhyd_mphys(7)
     type(c_ptr) :: ppt
  end type kidmp_kid_columns

  ! include/kidmp.h :: kidmp_wrf_fields, (i,k,j) arrays as c_loc of (ims:ime,kms:kme,jms:jme) arrays; ni, nk, nj are the memory
  ! dimensions (kidmp_mp_gt_driver steps the whole box: a host with halos or kme = kte+1 uses kidmp_mp_gt_driver_tile)
  type, bind(C) :: kidmp_wrf_fields
     integer(c_int) :: ni, nk, nj
     type(c_ptr) :: qv, qc, qr, qi, qs, qg, ni_, nr, th, pii, p, dz
     type(c_ptr) :: rainnc, rainncv, sr, snownc, snowncv, graupelnc, graupelncv
     type(c_ptr) :: re_cloud, re_ice, re_snow
  end type kidmp_wrf_fields
  ! mp_gt_driver's optional aerosol arguments (M:807-832) for is_aerosol_aware = .true. (M:28)
  type, bind(C) :: kidmp_wrf_aerosols
     type(c_ptr) :: nc, nwfa, nifa, w, nwfa2d
  end type kidmp_wrf_aerosols
  ! include/kidmp.h :: kidmp_wrf_tile, the tile to step inside the memory box of kidmp_wrf_fields (0-based offsets, extents).
  ! A WRF / MPAS caller passes the memory dimensions in kidmp_wrf_fields and its tile here:
  !   w%ni = ime-ims+1;  w%nk = kme-kms+1;  w%nj = jme-jms+1          (c_loc of the (ims:ime,kms:kme,jms:jme) arrays)
  !   t%i0 = its-ims;    t%ni = ite-its+1
  !   t%k0 = kts-kms;    t%nk = kte-kts+1                              (kme = kte+1: the spare top level stays out)
  !   t%j0 = jts-jms;    t%nj = jte-jts+1
  ! The call reads and writes only the tile, so the OpenMP tiles of one patch may step at the same time (one handle each).
  type, bind(C) :: kidmp_wrf_tile
     integer(c_int) :: i0, ni, k0, nk, j0, nj
  end type kidmp_wrf_tile

  interface
     integer(c_int) function kidmp_init(cfg, handle) bind(C, name='kidmp_init')
       import :: c_int, c_ptr, kidmp_config
       type(kidmp_config), intent(in) :: cfg
       type(c_ptr), intent(out) :: handle
     end function kidmp_init
     integer(c_int) function kidmp_kid_interface(handle, cols, dt, p0, r_on_cp) bind(C, name='kidmp_kid_interface')
       import :: c_int, c_ptr, c_float, kidmp_kid_columns
       type(c_ptr), value :: handle
       type(kidmp_kid_columns), intent(in) :: cols
       real(c_float), value :: dt, p0, r_on_cp
     end function kidmp_kid_interface
     type(c_ptr) function kidmp_last_error(handle) bind(C, name='kidmp_last_error')
       import :: c_ptr
       type(c_ptr), value :: handle
     end function kidmp_last_error
     integer(c_int) function kidmp_finalize(handle) bind(C, name='kidmp_finalize')
       import :: c_int, c_ptr
       type(c_ptr), value :: handle
     end function kidmp_finalize
     ! the 36 process rates that mp_thompson saves with save_dg (M:2963-3120): the handle keeps them, the host fetches them
     integer(c_int) function kidmp_enable_rates(handle, on) bind(C, name='kidmp_enable_rates')
       import :: c_int, c_ptr
       type(c_ptr), value :: handle
       integer(c_int), value :: on
     end function kidmp_enable_rates
     integer(c_int) function kidmp_get_rates(handle, layout, rates) bind(C, name='kidmp_get_rates')
       import :: c_int, c_ptr, c_float
       type(c_ptr), value :: handle
       integer(c_int), value :: layout
       real(c_float), intent(out) :: rates(*)
     end function kidmp_get_rates
     ! tuning knobs that never change a result, e.g. kidmp_set_option(handle, 'chunk'//c_null_char, 262144_c_int)
     integer(c_int) function kidmp_set_option(handle, name, value) bind(C, name='kidmp_set_option')
       import :: c_int, c_ptr, c_char
       type(c_ptr), value :: handle
       character(kind=c_char), intent(in) :: name(*)
       integer(c_int), value :: value
     end function kidmp_set_option
     ! the WRF / MPAS shape of the same step (mp_gt_driver, M:806-1143); KiD itself does not call it
     integer(c_int) function kidmp_mp_gt_driver(handle, w, dt_in) bind(C, name='kidmp_mp_gt_driver')
       import :: c_int, c_ptr, c_float, kidmp_wrf_fields
       type(c_ptr), value :: handle
       type(kidmp_wrf_fields), intent(in) :: w
       real(c_float), value :: dt_in
     end function kidmp_mp_gt_driver
     ! ... and with is_aerosol_aware = .true. (prognostic nc, nwfa, nifa; w; surface emission nwfa2d)
     integer(c_int) function kidmp_mp_gt_driver_aero(handle, w, ae, dt_in) bind(C, name='kidmp_mp_gt_driver_aero')
       import :: c_int, c_ptr, c_float, kidmp_wrf_fields, kidmp_wrf_aerosols
       type(c_ptr), value :: handle
       type(kidmp_wrf_fields), intent(in) :: w
       type(kidmp_wrf_aerosols), intent(in) :: ae
       real(c_float), value :: dt_in
     end function kidmp_mp_gt_driver_aero
     ! one tile of the memory box, host arrays; ae = c_null_ptr: is_aerosol_aware = .false., else c_loc of a kidmp_wrf_aerosols
     integer(c_int) function kidmp_mp_gt_driver_tile(handle, w, t, ae, dt_in) bind(C, name='kidmp_mp_gt_driver_tile')
       import :: c_int, c_ptr, c_float, kidmp_wrf_fields, kidmp_wrf_tile
       type(c_ptr), value :: handle
       type(kidmp_wrf_fields), intent(in) :: w
       type(kidmp_wrf_tile), intent(in) :: t
       type(c_ptr), value :: ae
       real(c_float), value :: dt_in
     end function kidmp_mp_gt_driver_tile
     ! ... the same on device arrays (e.g. OpenACC / CUDA Fortran device data), enqueued on `stream` (c_null_ptr = the handle's)
     integer(c_int) function kidmp_mp_gt_driver_tile_device(handle, w, t, ae, dt_in, stream) &
          bind(C, name='kidmp_mp_gt_driver_tile_device')
       import :: c_int, c_ptr, c_float, kidmp_wrf_fields, kidmp_wrf_tile
       type(c_ptr), value :: handle
       type(kidmp_wrf_fields), intent(in) :: w
       type(kidmp_wrf_tile), intent(in) :: t
       type(c_ptr), value :: ae
       real(c_float), value :: dt_in
       type(c_ptr), value :: stream
     end function kidmp_mp_gt_driver_tile_device
  end interface

  !Logical switches
  logical :: micro_unset=.True.
  integer:: ih, imom
  character(max_char_len) :: name, units
  type(c_ptr), save :: kidmp_handle = c_null_ptr
  character(kind=c_char, len=64), target, save :: cache_path = 'run_data/kidmp_tables.bin'//c_null_char

  ! switch for the per-level process-rate diagnostics of M:2963-3120 (36 rates x nz x nx floats back per call)
  logical :: save_process_rates = .true.
  integer, save :: kidmp_ndev = 1                 ! set > 1 before the first call to spread the nx columns over several GPUs
  ! the rates in the order of kidmp_rate_names(): 30 ice-phase rates, then the 6 warm ones (the reference's order)
  character(7), parameter :: rate_name(36) = (/ 'pri_inu', 'pri_ide', 'prs_ide', 'prs_sde', 'prg_gde', 'pri_wfz', 'prs_scw', &
       'prg_scw', 'prg_gcw', 'pri_ihm', 'pri_rfz', 'prs_iau', 'prs_sci', 'pri_rci', 'pni_inu', 'pni_ihm', 'pni_wfz', 'pni_rfz', &
       'pni_ide', 'pni_iau', 'pni_sci', 'pni_rci', 'prr_sml', 'prr_gml', 'pnr_rcs', 'pnr_rcg', 'pnr_rci', 'pnr_sml', 'pnr_gml', &
       'pnr_rfz', 'prr_wau', 'prr_rcw', 'prv_rev', 'pnr_wau', 'pnr_rev', 'pnr_rcr' /)

  ! order of the hydrometeor planes handed to the library: (ih, imom) of hydrometeors(k,i,ih)%moments(1,imom)
  integer, parameter :: plane_ih(7)   = (/1, 2, 2, 3, 3, 4, 5/)   ! cloud, rain, rain, ice, ice, snow, graupel
  integer, parameter :: plane_imom(7) = (/1, 1, 2, 1, 2, 1, 1/)   ! mass, mass, number, mass, number, mass, mass

contains

  Subroutine mphys_thompson09_interfacen

    real(c_float), target, save, allocatable :: hyd(:,:,:), hyd_adv(:,:,:), hyd_div(:,:,:), hyd_mphys(:,:,:)
    real(c_float), target, save, allocatable :: th(:,:), th_adv(:,:), th_div(:,:), ex(:,:), q(:,:), q_adv(:,:), q_div(:,:)
    real(c_float), target, save, allocatable :: dth_mphys(:,:), dq_mphys(:,:), ppt(:,:), dzc(:), rates(:,:,:)
    integer :: r, r0
    real :: pptrain_2d(nx), pptsnow_2d(nx), pptgraul_2d(nx), pptice_2d(nx), pptrain_2d_prof(nz,nx)
    type(kidmp_config) :: cfg
    type(kidmp_kid_columns) :: c
    integer :: i, k, m, np, rc

    ! Initialise microphysics (replaces `call thompson_init`, I:100-103)
    if (micro_unset) then
       cfg%set_Nc = set_Nc
       cfg%iiwarm = merge(1, 0, iiwarm)
       cfg%l_sediment = merge(1, 0, l_sediment)
       cfg%wp_double = merge(1, 0, kind(1.0) == kind(1.0d0))
       cfg%device = 0
       cfg%reuse_tables = merge(1, 0, l_reuse_thompson_lookup)
       cfg%table_cache_path = c_loc(cache_path)
       cfg%ndev = kidmp_ndev
       cfg%device_ids = c_null_ptr
       rc = kidmp_init(cfg, kidmp_handle)
       if (rc /= 0) then
          print *, 'kidmp_init failed'      ! text: kidmp_last_error(c_null_ptr)
          stop 1
       end if
       allocate(hyd(nz,nx,7), hyd_adv(nz,nx,7), hyd_div(nz,nx,7), hyd_mphys(nz,nx,7))
       allocate(th(nz,nx), th_adv(nz,nx), th_div(nz,nx), ex(nz,nx), q(nz,nx), q_adv(nz,nx), q_div(nz,nx))
       allocate(dth_mphys(nz,nx), dq_mphys(nz,nx), ppt(nx,4), dzc(nz))
       if (save_process_rates) then
          allocate(rates(nz,nx,36))
          rc = kidmp_enable_rates(kidmp_handle, 1_c_int)
       end if
       micro_unset=.False.
    end if

    ! pack KiD's derived-type state into plain (k,i) planes; the algebra of I:59-95 runs on the device
    np = 7
    if (iiwarm) np = 3
    do i=1,nx
       do k=1,nz
          th(k,i) = theta(k,i); th_adv(k,i) = dtheta_adv(k,i); th_div(k,i) = dtheta_div(k,i)
          ex(k,i) = exner(k,i)
          q(k,i) = qv(k,i); q_adv(k,i) = dqv_adv(k,i); q_div(k,i) = dqv_div(k,i)
          do m=1,np
             hyd(k,i,m)     = hydrometeors(k,i,plane_ih(m))%moments(1,plane_imom(m))
             hyd_adv(k,i,m) = dhydrometeors_adv(k,i,plane_ih(m))%moments(1,plane_imom(m))
             hyd_div(k,i,m) = dhydrometeors_div(k,i,plane_ih(m))%moments(1,plane_imom(m))
          end do
       end do
    end do
    dzc(:) = dz(:)

    c%nx = nx; c%nz = nz
    c%theta = c_loc(th); c%dtheta_adv = c_loc(th_adv); c%dtheta_div = c_loc(th_div); c%exner = c_loc(ex)
    c%qv = c_loc(q); c%dqv_adv = c_loc(q_adv); c%dqv_div = c_loc(q_div); c%dz = c_loc(dzc)
    do m=1,7
       if (m <= np) then
          c%hyd(m) = c_loc(hyd(1,1,m)); c%dhyd_adv(m) = c_loc(hyd_adv(1,1,m)); c%dhyd_div(m) = c_loc(hyd_div(1,1,m))
          c%dhyd_mphys(m) = c_loc(hyd_mphys(1,1,m))
       else
          c%hyd(m) = c_null_ptr; c%dhyd_adv(m) = c_null_ptr; c%dhyd_div(m) = c_null_ptr; c%dhyd_mphys(m) = c_null_ptr
       end if
    end do
    c%dtheta_mphys = c_loc(dth_mphys); c%dqv_mphys = c_loc(dq_mphys); c%ppt = c_loc(ppt)

    ! gather + mp_thompson for every column + back out tendencies (I:54-246), on the GPU
    rc = kidmp_kid_interface(kidmp_handle, c, real(dt, c_float), real(p0, c_float), real(r_on_cp, c_float))
    if (rc /= 0) then
       print *, 'kidmp_kid_interface failed'
       stop 1
    end if

    do i=1,nx
       do k=1,nz
          dtheta_mphys(k,i) = dth_mphys(k,i)
          dqv_mphys(k,i) = dq_mphys(k,i)
          do m=1,np
             dhydrometeors_mphys(k,i,plane_ih(m))%moments(1,plane_imom(m)) = hyd_mphys(k,i,m)
          end do
       end do
    end do

    ! the per-level process rates that mp_thompson itself saves (M:2963-3120): 36 save_dg calls per level, in the
    ! reference's order (column by column, level by level; the 30 ice-phase rates only when .not. iiwarm), with the
    ! (k, value) form for a single column and the (k, i, value) form otherwise
    if (save_process_rates) then
       rc = kidmp_get_rates(kidmp_handle, 0_c_int, rates)        ! KIDMP_K_FASTEST: rates(k,i,r)
       if (rc /= 0) then
          print *, 'kidmp_get_rates failed'
          stop 1
       end if
       r0 = 1
       if (iiwarm) r0 = 31
       do i=1,nx
          do k=1,nz
             do r=r0,36
                if (nx == 1) then
                   call save_dg(k, rates(k,i,r), rate_name(r), i_dgtime, units='/kg/s', dim='z')
                else
                   call save_dg(k, i, rates(k,i,r), rate_name(r), i_dgtime, units='/kg/s', dim='z,x')
                end if
             end do
          end do
       end do
    end if

    ! diagnostics exactly as the reference saves them (I:155-192, I:248-308); ppt(:,1..4) = rain, ice, snow, graupel
    pptrain_2d(:) = ppt(:,1); pptice_2d(:) = ppt(:,2); pptsnow_2d(:) = ppt(:,3); pptgraul_2d(:) = ppt(:,4)
    pptrain_2d_prof(:,:) = 0.0          ! never assigned in the reference (I:191 is commented out): zeros (U3)
    imom=1
    if (nx == 1) then
       ih=2
       name='surface_ppt_for_'//trim(h_names(ih)); units=trim(mom_units(imom))//' m'
       call save_dg(pptrain_2d(1), name, i_dgtime,  units, dim='time')
       ih=3
       name='surface_ppt_for_'//trim(h_names(ih)); units=trim(mom_units(imom))//' m'
       call save_dg(pptice_2d(1), name, i_dgtime,  units, dim='time')
       ih=4
       name='surface_ppt_for_'//trim(h_names(ih)); units=trim(mom_units(imom))//' m'
       call save_dg(pptsnow_2d(1), name, i_dgtime,  units, dim='time')
       ih=5
       name='surface_ppt_for_'//trim(h_names(ih)); units=trim(mom_units(imom))//' m'
       call save_dg(pptgraul_2d(1), name, i_dgtime,  units, dim='time')
       name='total_surface_ppt'; units=trim(mom_units(imom))//' m'
       call save_dg((pptice_2d(1)+pptrain_2d(1)+pptsnow_2d(1)+pptgraul_2d(1))/nx, name, i_dgtime, units, dim='time')
    else
       ih=2
       name='surface_ppt_for_'//trim(h_names(ih)); units=trim(mom_units(imom))//' m'
       call save_dg(pptrain_2d/nx, name, i_dgtime,  units, dim='time')
       call save_dg(pptrain_2d, name, i_dgtime,  units, dim='time')
       ih=3
       name='surface_ppt_for_'//trim(h_names(ih)); units=trim(mom_units(imom))//' m'
       call save_dg(pptice_2d/nx, name, i_dgtime,  units, dim='time')
       call save_dg(pptice_2d, name, i_dgtime,  units, dim='time')
       ih=4
       name='surface_ppt_for_'//trim(h_names(ih)); units=trim(mom_units(imom))//' m'
       call save_dg(pptsnow_2d/nx, name, i_dgtime,  units, dim='time')
       call save_dg(pptsnow_2d, name, i_dgtime,  units, dim='time')
       ih=5
       name='surface_ppt_for_'//trim(h_names(ih)); units=trim(mom_units(imom))//' m'
       call save_dg(pptgraul_2d/nx, name, i_dgtime,  units, dim='time')
       call save_dg(pptgraul_2d, name, i_dgtime,  units, dim='time')
       name='total_surface_ppt'; units=trim(mom_units(imom))//' m'
       call save_dg((pptice_2d+pptrain_2d+pptsnow_2d+pptgraul_2d)/nx, name, i_dgtime, units, dim='time')
       call save_dg((pptice_2d+pptrain_2d+pptsnow_2d+pptgraul_2d), name, i_dgtime, units, dim='time')
       name='total_ppt_level'; units=trim(mom_units(imom))//' m'
       call save_dg(pptrain_2d_prof, name, i_dgtime,  units, dim='z,x')
    endif

  end Subroutine mphys_thompson09_interfacen

  ! BASELINE.json spells the entry point without the trailing n; keep both names callable
  Subroutine mphys_thompson09_interface
    call mphys_thompson09_interfacen
  end Subroutine mphys_thompson09_interface

end module mphys_thompson09n
