!--- rtb200_shim: ISO_C_BINDING bridge between the unchanged FTTE driver (equiSources.f90) and librtb200.so.
!--- The octree (zoneType, definitionsModule.f90:163-182) has pointer components and is not interoperable, so the
!--- shim flattens the leaves in writeCell order (equiSources.f90:4044-4079), calls the C-ABI of include/rtb200.h and
!--- scatters the results back into the same cells.  A non-zero status reproduces the reference's `write; stop`.
!--- NOTE: no Fortran compiler exists in the build image of this repository; this file is syntax-reviewed only.
module rtb200_shim

  use iso_c_binding
  use definitions

  implicit none
  type(c_ptr), save :: rtbContext = c_null_ptr
  integer(c_int), save :: rtbGpus = 1          ! GPUs of this node the library drives (rtbInit); one process, one handle
  integer(c_int64_t), save :: rtbLeaves = 0
  integer(c_int8_t), dimension(:), allocatable, target, save :: flatLevel
  real(c_double), dimension(:), allocatable, target, save :: flatHI, flatHeI, flatHeII, flatRho, flatAbun2, &
       flatJ1, flatJ2, flatJ3
  integer(c_int64_t), save :: icursor
  ! point sources: six rate fields
  real(c_double), dimension(:), allocatable, target, save :: flatK24, flatK25, flatK26, flatC24, flatC25, flatC26

  interface
     integer(c_int) function rtb200_create(device, ctx) bind(C, name='rtb200_create')
       import :: c_int, c_ptr
       integer(c_int), value :: device
       type(c_ptr) :: ctx
     end function rtb200_create
     ! one handle for `ngpus` devices of this node (devices = c_null_ptr: 0..ngpus-1); every call below accepts it and
     ! shards the directions / sources inside the library (include/rtb200.h, "Device groups")
     integer(c_int) function rtb200_create_multi(ngpus, devices, ctx) bind(C, name='rtb200_create_multi')
       import :: c_int, c_ptr
       integer(c_int), value :: ngpus
       type(c_ptr), value :: devices
       type(c_ptr) :: ctx
     end function rtb200_create_multi
     integer(c_int) function rtb200_destroy(ctx) bind(C, name='rtb200_destroy')
       import :: c_int, c_ptr
       type(c_ptr), value :: ctx
     end function rtb200_destroy
     integer(c_int) function rtb200_grid_set(ctx, nx, nleaf, level, HI, HeI, HeII, rho, abun2, boxSize) &
          bind(C, name='rtb200_grid_set')
       import :: c_int, c_int64_t, c_ptr, c_double
       type(c_ptr), value :: ctx
       integer(c_int), value :: nx
       integer(c_int64_t), value :: nleaf
       type(c_ptr), value :: level, HI, HeI, HeII, rho, abun2
       real(c_double), value :: boxSize
     end function rtb200_grid_set
     integer(c_int) function rtb200_grid_update_species(ctx, HI, HeI, HeII) bind(C, name='rtb200_grid_update_species')
       import :: c_int, c_ptr
       type(c_ptr), value :: ctx, HI, HeI, HeII
     end function rtb200_grid_update_species
     integer(c_int) function rtb200_grid_set_emission(ctx, eta) bind(C, name='rtb200_grid_set_emission')
       import :: c_ptr, c_int
       type(c_ptr), value :: ctx, eta
     end function rtb200_grid_set_emission
     integer(c_int) function rtb200_grid_set_scattering(ctx, sigma, maxIterations, tolerance) &
          bind(C, name='rtb200_grid_set_scattering')
       import :: c_ptr, c_int, c_int32_t, c_double
       type(c_ptr), value :: ctx, sigma
       integer(c_int32_t), value :: maxIterations
       real(c_double), value :: tolerance
     end function rtb200_grid_set_scattering
     integer(c_int) function rtb200_last_scattering(ctx, iterations, residual) bind(C, name='rtb200_last_scattering')
       import :: c_ptr, c_int, c_int32_t, c_double
       type(c_ptr), value :: ctx
       integer(c_int32_t), intent(out) :: iterations
       real(c_double), intent(out) :: residual
     end function rtb200_last_scattering
     integer(c_int) function rtb200_grid_set_dust(ctx, dustApproximation, betaDust, albedo, maxIterations, tolerance) &
          bind(C, name='rtb200_grid_set_dust')
       import :: c_ptr, c_int, c_int32_t, c_double
       type(c_ptr), value :: ctx, betaDust, albedo
       integer(c_int), value :: dustApproximation
       integer(c_int32_t), value :: maxIterations
       real(c_double), value :: tolerance
     end function rtb200_grid_set_dust
     integer(c_int) function rtb200_uvb_dust_beta(nfreq, freqdel, alpha, aDust, betaDust) bind(C, name='rtb200_uvb_dust_beta')
       import :: c_ptr, c_int, c_double
       integer(c_int), value :: nfreq
       real(c_double), value :: freqdel
       type(c_ptr), value :: alpha, aDust, betaDust
     end function rtb200_uvb_dust_beta
     integer(c_int) function rtb200_diffuse(ctx, nAngularLevel, uvb, beta, rays, nrays, J1, J2, J3, nseg) &
          bind(C, name='rtb200_diffuse')
       import :: c_int, c_int32_t, c_ptr
       type(c_ptr), value :: ctx
       integer(c_int), value :: nAngularLevel
       type(c_ptr), value :: uvb, beta, rays
       integer(c_int32_t), value :: nrays
       type(c_ptr), value :: J1, J2, J3, nseg
     end function rtb200_diffuse
     integer(c_int) function rtb200_chemistry_tables(ctx, nratec, logtem0, logtem9, dlogtem, k1a, k2a, k3a, k4a, k5a, k6a) &
          bind(C, name='rtb200_chemistry_tables')
       import :: c_int, c_ptr, c_double
       type(c_ptr), value :: ctx
       integer(c_int), value :: nratec
       real(c_double), value :: logtem0, logtem9, dlogtem
       type(c_ptr), value :: k1a, k2a, k3a, k4a, k5a, k6a
     end function rtb200_chemistry_tables
     integer(c_int) function rtb200_chemistry_temperature(ctx, tgas) bind(C, name='rtb200_chemistry_temperature')
       import :: c_int, c_ptr
       type(c_ptr), value :: ctx, tgas
     end function rtb200_chemistry_temperature
     integer(c_int) function rtb200_chemistry_device(ctx, rates_device, J_device, ksi, uniform, maxChange, stream) &
          bind(C, name='rtb200_chemistry_device')
       import :: c_int, c_ptr
       type(c_ptr), value :: ctx, rates_device, J_device, ksi, uniform, maxChange, stream
     end function rtb200_chemistry_device
     integer(c_int) function rtb200_compute_mass(ctx, neutralMass, totalMass, stream) bind(C, name='rtb200_compute_mass')
       import :: c_int, c_ptr, c_double
       type(c_ptr), value :: ctx
       real(c_double), intent(out) :: neutralMass, totalMass   ! neutralHydrogenMass, totalHydrogenMass [msun]
       type(c_ptr), value :: stream
     end function rtb200_compute_mass
     integer(c_int) function rtb200_grid_get_species(ctx, HI, HeI, HeII) bind(C, name='rtb200_grid_get_species')
       import :: c_int, c_ptr
       type(c_ptr), value :: ctx, HI, HeI, HeII
     end function rtb200_grid_get_species
     integer(c_int) function rtb200_point(ctx, nWave, wavelength, lum, metallicity, coefSpectrum, aDust, &
          dustApproximation, maxPixelLevel, nsrc, srcLeaf, srcWeight, k24, k25, k26, c24, c25, c26, &
          ndotRemaining, ndotBoundary, ndotDust, ndotSpectrum, highestPixelLevel, nseg) bind(C, name='rtb200_point')
       import :: c_int, c_int32_t, c_ptr, c_double
       type(c_ptr), value :: ctx
       integer(c_int), value :: nWave
       type(c_ptr), value :: wavelength, lum, metallicity
       real(c_double), value :: coefSpectrum
       type(c_ptr), value :: aDust
       integer(c_int), value :: dustApproximation, maxPixelLevel
       integer(c_int32_t), value :: nsrc
       type(c_ptr), value :: srcLeaf, srcWeight, k24, k25, k26, c24, c25, c26
       type(c_ptr), value :: ndotRemaining, ndotBoundary, ndotDust, ndotSpectrum, highestPixelLevel, nseg
     end function rtb200_point
  end interface

contains

  subroutine rtbCheck(status, where)
    integer(c_int), intent(in) :: status
    character(len=*), intent(in) :: where
    if (status.ne.0) then
       write(*,*) 'rtb200 error in ', where, ' status =', status
       stop
    endif
  end subroutine rtbCheck

  ! depth-first leaf order of writeCell (equiSources.f90:4044-4079): children i, j, k
  recursive subroutine countLeaves(currentCell, n)
    type(zoneType) :: currentCell
    integer(c_int64_t), intent(inout) :: n
    integer :: i, j, k
    if (currentCell%refined) then
       do i = 1, 2
          do j = 1, 2
             do k = 1, 2
                call countLeaves(currentCell%cell(i,j,k), n)
             enddo
          enddo
       enddo
    else
       n = n + 1
    endif
  end subroutine countLeaves

  recursive subroutine flattenCell(currentCell, level)
    type(zoneType) :: currentCell
    integer, intent(in) :: level
    integer :: i, j, k
    if (currentCell%refined) then
       do i = 1, 2
          do j = 1, 2
             do k = 1, 2
                call flattenCell(currentCell%cell(i,j,k), level+1)
             enddo
          enddo
       enddo
    else
       icursor = icursor + 1
       flatLevel(icursor) = int(level, c_int8_t)
       flatHI(icursor) = currentCell%HI
       flatHeI(icursor) = currentCell%HeI
       flatHeII(icursor) = currentCell%HeII
       flatRho(icursor) = currentCell%rho
       flatAbun2(icursor) = currentCell%abun2
    endif
  end subroutine flattenCell

  recursive subroutine scatterJ(currentCell)
    type(zoneType) :: currentCell
    integer :: i, j, k
    if (currentCell%refined) then
       do i = 1, 2
          do j = 1, 2
             do k = 1, 2
                call scatterJ(currentCell%cell(i,j,k))
             enddo
          enddo
       enddo
    else
       icursor = icursor + 1
       currentCell%Jmean1 = flatJ1(icursor)
       currentCell%Jmean2 = flatJ2(icursor)
       currentCell%Jmean3 = flatJ3(icursor)
    endif
  end subroutine scatterJ

  ! optional, before rtbSetGrid: how many GPUs of this node to use (default: environment variable RTB200_GPUS, else 1).
  ! The driver stays ONE serial process; the library opens all devices behind one handle.
  subroutine rtbInit(ngpus)
    integer, intent(in) :: ngpus
    if (c_associated(rtbContext)) then
       call rtbCheck(rtb200_destroy(rtbContext), 'rtb200_destroy')
       rtbContext = c_null_ptr
    endif
    rtbGpus = int(max(1, ngpus), c_int)
  end subroutine rtbInit

  ! once, after the octree is built (equiSources.f90:628) -- and again whenever its topology changes
  subroutine rtbSetGrid(nx, ny, nz)
    integer, intent(in) :: nx, ny, nz
    integer :: i, j, k, ios, envGpus
    character(len=16) :: envValue
    if (nx.ne.ny .or. nx.ne.nz) then
       write(*,*) 'rtb200: cubic base grid required'
       stop
    endif
    if (.not.c_associated(rtbContext)) then
       call get_environment_variable('RTB200_GPUS', envValue, status=ios)
       if (ios.eq.0) then
          read(envValue, *, iostat=ios) envGpus
          if (ios.eq.0 .and. envGpus.ge.1) rtbGpus = int(envGpus, c_int)
       endif
       if (rtbGpus.gt.1) then
          call rtbCheck(rtb200_create_multi(rtbGpus, c_null_ptr, rtbContext), 'rtb200_create_multi')
       else
          call rtbCheck(rtb200_create(0_c_int, rtbContext), 'rtb200_create')
       endif
    endif
    rtbLeaves = 0
    do i = 1, nx
       do j = 1, ny
          do k = 1, nz
             call countLeaves(baseGrid%cell(i,j,k), rtbLeaves)
          enddo
       enddo
    enddo
    if (allocated(flatLevel)) deallocate(flatLevel, flatHI, flatHeI, flatHeII, flatRho, flatAbun2, flatJ1, flatJ2, flatJ3)
    allocate(flatLevel(rtbLeaves), flatHI(rtbLeaves), flatHeI(rtbLeaves), flatHeII(rtbLeaves), flatRho(rtbLeaves), &
         flatAbun2(rtbLeaves), flatJ1(rtbLeaves), flatJ2(rtbLeaves), flatJ3(rtbLeaves))
    icursor = 0
    do i = 1, nx
       do j = 1, ny
          do k = 1, nz
             call flattenCell(baseGrid%cell(i,j,k), 0)
          enddo
       enddo
    enddo
    call rtbCheck(rtb200_grid_set(rtbContext, int(nx, c_int), rtbLeaves, c_loc(flatLevel), c_loc(flatHI), &
         c_loc(flatHeI), c_loc(flatHeII), c_loc(flatRho), c_loc(flatAbun2), real(physicalBoxSize, c_double)), &
         'rtb200_grid_set')
  end subroutine rtbSetGrid

  ! replaces equiSources.f90:1372-1808 (runUVBTransfer block) inside the outer loop
  subroutine rtbDiffuse(nx, ny, nz)
    integer, intent(in) :: nx, ny, nz
    integer :: i, j, k
    real(c_double), dimension(3), target :: uvb
    real(c_double), dimension(9), target :: beta
    uvb = (/ uvb1, uvb2, uvb3 /)
    ! [group][beta24, beta26, beta25] as computeOpacities uses them (equiSources.f90:4974-4977)
    beta = (/ group1%beta24, group1%beta26, group1%beta25, &
              group2%beta24, group2%beta26, group2%beta25, &
              group3%beta24, group3%beta26, group3%beta25 /)
    ! chemistry changed HI, HeI, HeII since the last call (equiSources.f90:3671-3673)
    icursor = 0
    do i = 1, nx
       do j = 1, ny
          do k = 1, nz
             call flattenCell(baseGrid%cell(i,j,k), 0)
          enddo
       enddo
    enddo
    call rtbCheck(rtb200_grid_update_species(rtbContext, c_loc(flatHI), c_loc(flatHeI), c_loc(flatHeII)), &
         'rtb200_grid_update_species')
    call rtbCheck(rtb200_diffuse(rtbContext, int(nAngularLevel, c_int), c_loc(uvb), c_loc(beta), c_null_ptr, &
         0_c_int32_t, c_loc(flatJ1), c_loc(flatJ2), c_loc(flatJ3), c_null_ptr), 'rtb200_diffuse')
    icursor = 0
    do i = 1, nx
       do j = 1, ny
          do k = 1, nz
             call scatterJ(baseGrid%cell(i,j,k))
          enddo
       enddo
    enddo
  end subroutine rtbDiffuse

  ! ---- point sources ---------------------------------------------------------------------------------------

  recursive subroutine scatterRates(currentCell)
    type(zoneType) :: currentCell
    integer :: i, j, k
    if (currentCell%refined) then
       do i = 1, 2
          do j = 1, 2
             do k = 1, 2
                call scatterRates(currentCell%cell(i,j,k))
             enddo
          enddo
       enddo
    else
       icursor = icursor + 1
       currentCell%krate24 = flatK24(icursor)
       currentCell%krate25 = flatK25(icursor)
       currentCell%krate26 = flatK26(icursor)
       currentCell%crate24 = flatC24(icursor)
       currentCell%crate25 = flatC25(icursor)
       currentCell%crate26 = flatC26(icursor)
    endif
  end subroutine scatterRates

  ! Leaf numbers (0-based, writeCell order) of the stars' host cells in O(leaves + stars): one walk writes every
  ! leaf's number into its krate24 field -- free at this point, setZeroRates (equiSources.f90:1246) has just cleared the
  ! rate fields and scatterRates overwrites them below -- and star%hostCell (:753-756) reads it back.
  recursive subroutine markLeafNumbers(currentCell)
    type(zoneType) :: currentCell
    integer :: i, j, k
    if (currentCell%refined) then
       do i = 1, 2
          do j = 1, 2
             do k = 1, 2
                call markLeafNumbers(currentCell%cell(i,j,k))
             enddo
          enddo
       enddo
    else
       currentCell%krate24 = real(icursor, kind=RealKind)   ! exact: leaf numbers are below 2**31
       icursor = icursor + 1
    endif
  end subroutine markLeafNumbers

  ! replaces equiSources.f90:1256-1370 (runStellarTransfer block): all sources with weight > 0 in one call.
  ! iSpectrum / coefSpectrum are the driver's locals computed at :1236-1242.
  subroutine rtbPoint(nx, ny, nz, iSpectrum, coefSpectrum, maxPixelLevel, nStarsSpecificAge)
    integer, intent(in) :: nx, ny, nz, iSpectrum, maxPixelLevel, nStarsSpecificAge
    real(kind=RealKind), intent(in) :: coefSpectrum
    integer :: i, j, k, iStar, nsrc, iradius, im
    integer(c_int32_t), dimension(:), allocatable, target :: srcLeaf, srcWeight, highestLevel
    real(c_double), dimension(:,:), allocatable, target :: remaining, boundary, spectrum   ! (7,nsrc), (7,nsrc), (300,nsrc)
    real(c_double), dimension(:), allocatable, target :: dustEscape
    real(c_double), dimension(nWavelengths,2,nMetallicity), target :: lumPack   ! = C [5][2][nWave]
    real(c_double), dimension(5,7), target :: dustPack                         ! = C [7][5]
    real(c_double), dimension(nWavelengths), target :: wl
    real(c_double), dimension(nMetallicity), target :: met
    real(kind=RealKind) :: ndot1, fraction(7)

    if (allocated(flatK24)) then
       if (size(flatK24).ne.rtbLeaves) deallocate(flatK24, flatK25, flatK26, flatC24, flatC25, flatC26)
    endif
    if (.not.allocated(flatK24)) allocate(flatK24(rtbLeaves), flatK25(rtbLeaves), flatK26(rtbLeaves), &
         flatC24(rtbLeaves), flatC25(rtbLeaves), flatC26(rtbLeaves))
    icursor = 0
    do i = 1, nx
       do j = 1, ny
          do k = 1, nz
             call markLeafNumbers(baseGrid%cell(i,j,k))
          enddo
       enddo
    enddo
    nsrc = 0
    do iStar = 1, nStars
       if (star(iStar)%weight.gt.0) nsrc = nsrc + 1
    enddo
    allocate(srcLeaf(nsrc), srcWeight(nsrc), highestLevel(nsrc), remaining(7,nsrc), boundary(7,nsrc), &
         spectrum(300,nsrc), dustEscape(nsrc))
    nsrc = 0
    do iStar = 1, nStars
       if (star(iStar)%weight.gt.0) then
          nsrc = nsrc + 1
          srcLeaf(nsrc) = int(star(iStar)%hostCell%krate24, c_int32_t)
          srcWeight(nsrc) = star(iStar)%weight
       endif
    enddo
    do im = 1, nMetallicity
       lumPack(:,1,im) = specificLuminosity(im,iSpectrum,:)
       lumPack(:,2,im) = specificLuminosity(im,iSpectrum+1,:)
    enddo
    dustPack = transpose(a_smc)
    wl = wavelength
    met = metallicity
    ! absorber densities may have changed since rtbSetGrid (previous chemistry step)
    icursor = 0
    do i = 1, nx
       do j = 1, ny
          do k = 1, nz
             call flattenCell(baseGrid%cell(i,j,k), 0)
          enddo
       enddo
    enddo
    call rtbCheck(rtb200_grid_update_species(rtbContext, c_loc(flatHI), c_loc(flatHeI), c_loc(flatHeII)), &
         'rtb200_grid_update_species')
    flatK24 = 0.; flatK25 = 0.; flatK26 = 0.; flatC24 = 0.; flatC25 = 0.; flatC26 = 0.   ! setZeroRates (:1246)
    call rtbCheck(rtb200_point(rtbContext, int(nWavelengths, c_int), c_loc(wl), c_loc(lumPack), c_loc(met), &
         real(coefSpectrum, c_double), c_loc(dustPack), int(dustApproximation, c_int), int(maxPixelLevel, c_int), &
         int(nsrc, c_int32_t), c_loc(srcLeaf), c_loc(srcWeight), c_loc(flatK24), c_loc(flatK25), c_loc(flatK26), &
         c_loc(flatC24), c_loc(flatC25), c_loc(flatC26), c_loc(remaining), c_loc(boundary), c_loc(dustEscape), &
         c_loc(spectrum), c_loc(highestLevel), c_null_ptr), 'rtb200_point')
    icursor = 0
    do i = 1, nx
       do j = 1, ny
          do k = 1, nz
             call scatterRates(baseGrid%cell(i,j,k))
          enddo
       enddo
    enddo
    ! per-source escape fractions and the escaping spectrum (equiSources.f90:1342-1366)
    cosmicSpectrum = 0.
    nsrc = 0
    do iStar = 1, nStars
       if (star(iStar)%weight.gt.0) then
          nsrc = nsrc + 1
          ndot1 = float(star(iStar)%weight)
          do iradius = 1, 7
             if (boundary(iradius,nsrc).lt.1.) then
                fraction(iradius) = remaining(iradius,nsrc)/(ndot1-boundary(iradius,nsrc))
             else
                fraction(iradius) = 0.
             endif
          enddo
          cosmicSpectrum = cosmicSpectrum + float(star(iStar)%weight) * spectrum(:,nsrc)/(ndot1-boundary(7,nsrc))
          ! the driver's own line and format (equiSources.f90:1353-1357)
          write(*,1015) iStar, star(iStar)%level, &
               star(iStar)%hostCell%HI * mh / (psi * star(iStar)%hostCell%rho), &
               highestLevel(nsrc), fraction, star(iStar)%weight
       endif
    enddo
1015 format('src: ', i5, i3, es13.5, i3, 7f9.5, i8)
    cosmicSpectrum = cosmicSpectrum / float(nStarsSpecificAge)
    deallocate(srcLeaf, srcWeight, highestLevel, remaining, boundary, spectrum, dustEscape)
  end subroutine rtbPoint

  ! Emission coefficients per leaf (extension, DESIGN.md 4.6): eta(leaf, group) in the leaf order of rtbSetGrid, i.e.
  ! [3][nleaf] in C; the driver flattens its per-cell emissivities in the same writeCell pre-order as the species.
  ! Without the argument the emission is cleared.  Negative, NaN or Inf entries stop with RTB200_ERR_ARG.
  subroutine rtbSetEmission(eta)
    real(c_double), dimension(:,:), target, contiguous, intent(in), optional :: eta
    if (present(eta)) then
       call rtbCheck(rtb200_grid_set_emission(rtbContext, c_loc(eta)), 'rtb200_grid_set_emission')
    else
       call rtbCheck(rtb200_grid_set_emission(rtbContext, c_null_ptr), 'rtb200_grid_set_emission')
    endif
  end subroutine rtbSetEmission

  ! Isotropic scattering (extension, DESIGN.md 4.7): sigma(leaf, group) in 1/cm, in the leaf order of rtbSetGrid as
  ! rtbSetEmission.  The diffuse sweep then solves by source iteration, at most maxIterations sweeps, stopping once the
  ! relative change of J is <= tolerance (0: exactly maxIterations sweeps).  Without sigma the scattering is cleared.
  ! Negative, NaN or Inf entries, maxIterations < 1 or a negative tolerance stop with RTB200_ERR_ARG.
  subroutine rtbSetScattering(sigma, maxIterations, tolerance)
    real(c_double), dimension(:,:), target, contiguous, intent(in), optional :: sigma
    integer, intent(in) :: maxIterations
    real(c_double), intent(in) :: tolerance
    if (present(sigma)) then
       call rtbCheck(rtb200_grid_set_scattering(rtbContext, c_loc(sigma), int(maxIterations, c_int32_t), tolerance), &
            'rtb200_grid_set_scattering')
    else
       call rtbCheck(rtb200_grid_set_scattering(rtbContext, c_null_ptr, int(maxIterations, c_int32_t), tolerance), &
            'rtb200_grid_set_scattering')
    endif
  end subroutine rtbSetScattering

  ! sweeps done and the last residual of the latest diffuse call (0 / 0 without scattering)
  subroutine rtbScatteringStatus(iterations, residual)
    integer, intent(out) :: iterations
    real(c_double), intent(out) :: residual
    integer(c_int32_t) :: it
    call rtbCheck(rtb200_last_scattering(rtbContext, it, residual), 'rtb200_last_scattering')
    iterations = int(it)
  end subroutine rtbScatteringStatus

  ! Dust in the diffuse sweep (extension, DESIGN.md 4.8): the dust model of the point-source path (a_smc, dustModule.f90)
  ! as an opacity of the UV background, recomputed from the current species in every rtbDiffuse.  dustApproximation
  ! 1 / 2 as for the point sources, 0 clears it.  The band-mean dust cross-sections of the three groups come from
  ! alpha(3) and a_smc with the weights of uvbBetaTable (nfbins bins of frequencyBinWidth).  albedo(g) > 0 makes the
  ! dust scatter (source iteration, maxIterations / tolerance as rtbSetScattering; not together with rtbSetScattering).
  subroutine rtbSetDust(dustApproximation, albedo, maxIterations, tolerance)
    integer, intent(in) :: dustApproximation, maxIterations
    real(c_double), dimension(3), intent(in) :: albedo
    real(c_double), intent(in) :: tolerance
    real(c_double), dimension(3), target :: alphaC, betaDust, albedoC
    real(c_double), dimension(5,7), target :: dustPack                         ! = C [7][5]
    alphaC = real(alpha(1:3), c_double)
    dustPack = transpose(real(a_smc, c_double))
    albedoC = albedo
    call rtbCheck(rtb200_uvb_dust_beta(int(nfbins, c_int), real(frequencyBinWidth, c_double), c_loc(alphaC), &
         c_loc(dustPack), c_loc(betaDust)), 'rtb200_uvb_dust_beta')
    call rtbCheck(rtb200_grid_set_dust(rtbContext, int(dustApproximation, c_int), c_loc(betaDust), c_loc(albedoC), &
         int(maxIterations, c_int32_t), tolerance), 'rtb200_grid_set_dust')
  end subroutine rtbSetDust

end module rtb200_shim
