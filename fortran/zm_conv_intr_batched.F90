module zm_conv_intr_batched
!---------------------------------------------------------------------------------
! Batched (all chunks of a rank in one call) binding of zm_conv_tend / zm_conv_tend_2
! (NorESMhub/CAM-Nor-physics physics/zm_conv_intr.F90:390-951, 955-1028) to libzmconv_b200.so
! (include/zmconv_b200.h).  This is the entry a GPU needs: the per-chunk shim (zm_conv_shim.F90) feeds it 16
! columns per call.
!
! How it is used (INTEGRATION.md section 2): tphysbc's chunk loop (physpkg.F90:1147-1161, body :2808-2868) is
! split around convect_deep_tend.  Loop 1 runs every chunk up to dadadj_tend and calls zm_batch_gather; one call
! of zm_conv_tend_batched runs zm_convr -> physics_update -> zm_conv_evap -> momtran -> convtran1 for all chunks
! on the device; loop 2 calls zm_batch_scatter for its chunk (ptend_all, the dummy outputs of zm_conv_tend, the
! pbuf fields, the history diagnostics) and carries on with physics_update / check_energy_chng.
! zm_conv_tend_2_batched does the same for zm_conv_tend_2 (called from tphysac).
!
! Gathered mode (zm_batch_init(..., gathered=.true.)): the step returns the twenty (pcols,pver[p]) outputs as one
! record per convective column (zm_conv_tend_batch_gathered) instead of twenty dense rank-level arrays, and
! zm_batch_scatter writes each chunk's records into ptend_all (zeroed by physics_ptend_init) and into the dummy
! outputs and pbuf fields, which it zeroes first.  The outputs are the same; about a third of the bytes cross PCIe
! and host memory (INTEGRATION.md section 2).  zm_conv_tend_2 follows suit: zm_batch_gather_2 packs the convective
! columns of the constituents flagged convtran2 (and their pdeldry when one of them is dry), zm_conv_tend_2_batched
! transports those records (zm_conv_tend_2_batch_gathered) and zm_batch_scatter_2 scatters them into the ptend that
! physics_ptend_init has just zeroed.  The columns are ideep_b / lengath_b of this time step's zm_conv_tend_batched.
!
! The five GPTL timers of the reference (t_startf/t_stopf 'zm_convr', 'zm_conv_evap', 'momtran', 'convtran1',
! zm_conv_intr.F90:654-880, and 'convtran2', :1019-1025) cannot bracket host code any more -- the phases run
! back to back on the device -- so zm_batch_report_timers reads the device times of the phases back with
! zm_get_timers under the same names (zm_set_profiling(1) switches the event recording on) and writes them to
! the log; the wall-clock timers 'zm_conv_tend_batch' and 'zm_conv_tend_2_batch' bracket the calls.
!
! NOT COMPILED IN THIS REPOSITORY: the build image has no Fortran compiler.  tests/test_fortran_binding.py
! checks every bind(C) interface of this file and of zm_conv_shim.F90 against include/zmconv_b200.h with the C
! compiler: argument count, order (by name), types, const-ness, pass-by-value.
!---------------------------------------------------------------------------------
  use, intrinsic :: iso_c_binding
  use shr_kind_mod,    only: r8 => shr_kind_r8
  use ppgrid,          only: pcols, pver, pverp
  use physconst,       only: gravit, cpair
  use constituents,    only: pcnst, cnst_is_convtran1, cnst_is_convtran2, cnst_get_type_byind, cnst_get_ind
  use cam_abortutils,  only: endrun
  use cam_logfile,     only: iulog
  use cam_history,     only: outfld
  use perf_mod,        only: t_startf, t_stopf
  use phys_control,    only: cam_physpkg_is

  implicit none
  save
  private

  public :: zm_batch_init, zm_batch_gather, zm_conv_tend_batched, zm_batch_scatter
  public :: zm_batch_gather_2, zm_conv_tend_2_batched, zm_batch_scatter_2, zm_batch_report_timers

  ! ---- rank-level arrays: the chunks' (pcols,pver) fields back to back, [chunk][k][i] in C terms ----
  integer :: nchunks_b = 0
  integer(c_int),  allocatable :: ncol_b(:)
  real(c_double), allocatable, dimension(:,:,:) :: t_b, q_b, u_b, v_b, pmid_b, pdel_b, zm_b, cld_b        ! (pcols,pver,nchunks)
  real(c_double), allocatable, dimension(:,:,:) :: pint_b, zi_b                                            ! (pcols,pverp,nchunks)
  real(c_double), allocatable, dimension(:,:)   :: phis_b, pblh_b, tpert_b, landfrac_b, ps_b              ! (pcols,nchunks)
  real(c_double), allocatable, dimension(:,:,:) :: ptend_s_b, ptend_q_b, ptend_u_b, ptend_v_b, cme_b, zdu_b, &
                                                    ql_b, rprd_b, evapcdp_b, dlf_b, mu_b, md_b, du_b, eu_b, ed_b, dp_b, &
                                                    mu_out_b, md_out_b
  real(c_double), allocatable, dimension(:,:,:) :: mcon_b, pflx_b, flxprec_b, flxsnow_b
  real(c_double), allocatable, dimension(:,:)   :: rliq_b, rice_b, jctop_b, jcbot_b, prec_b, snow_b, dsubcld_b, cape_b, &
                                                    freqzm_b, pcont_b, pconb_b
  integer(c_int),  allocatable, dimension(:,:)   :: jt_b, maxg_b, ideep_b
  integer(c_int),  allocatable :: lengath_b(:)
  real(c_double), allocatable, dimension(:,:,:,:) :: q3_b, fracis_b, ptend_q3_b                            ! (pcols,pver,pcnst,nchunks)
  real(c_double), allocatable, dimension(:,:,:) :: pdeldry_b
  integer(c_int) :: doconvtran1(pcnst), doconvtran2(pcnst), cnst_is_dry(pcnst)
  ! history fields of zm_conv_tend (zm_conv_intr.F90:676-857): zm_convr's, zm_conv_evap's and momtran's own outputs,
  ! attached with zm_conv_tend_hist_fields; the momtran arrays are (pcols,pver,2,nchunks), component 1 = u, 2 = v
  real(c_double), allocatable, dimension(:,:,:) :: heat_b, qtnd_b, eurt_b, dif_b, dnlf_b, dnif_b, tend_s_b, &
                                                    snwprd_b, snwevmlt_b, ntprprd_b, ntsnprd_b, seten_b
  real(c_double), allocatable, dimension(:,:,:,:) :: pguall_b, pgdall_b, icwu_b, icwd_b
  ! zmconv_org: the organisation tracer state%q(:,:,ixorg) in, its tendency and column mean out (zm_conv.F90:421-423)
  logical :: org_on = .false.
  integer :: ixorg = -1
  real(c_double), allocatable, dimension(:,:,:) :: org_b, orgt_b, org2d_b
  ! gathered mode: the records of the convective columns, chunk after chunk (layout: include/zmconv_b200.h,
  ! zm_conv_tend_batch_gathered); rec_base_b(c) = sum(lengath_b(1:c-1)) is chunk c's first record
  logical :: gathered_on = .false.
  integer :: rec_len_b = 0
  real(c_double), allocatable :: rec_b(:)
  integer(c_long_long), allocatable :: rec_base_b(:)
  ! gathered mode, zm_conv_tend_2: the records of the nact2 constituents iact2 flagged convtran2; chunk c's block is
  ! g(lengath_b(c), pver, nact2) at nact2*pver*rec_base_b(c), its pdeldry(ideep(1:n),:) at pver*rec_base_b(c)
  integer :: nact2 = 0
  integer, allocatable :: iact2(:)
  logical :: dry2_any = .false.
  real(c_double), allocatable :: q2rec_b(:), fracis2rec_b(:), pdeldry2rec_b(:), dq2rec_b(:)

  interface
     integer(c_int) function zm_conv_tend_batch(nchunks, ncol, t, q, u, v, pmid, pint, pdel, zm, zi, phis, pblh, &
          tpert, landfrac, cld, ztodt, ptend_s, ptend_q, ptend_u, ptend_v, mcon, cme, pflx, zdu, rliq, rice, &
          jctop, jcbot, prec, snow, ql, rprd, evapcdp, flxprec, flxsnow, dlf, mu, md, du, eu, ed, dp, dsubcld, &
          jt, maxg, ideep, lengath, cape) bind(C, name='zm_conv_tend_batch')
       import :: c_int, c_double
       integer(c_int), value :: nchunks
       integer(c_int), intent(in) :: ncol(*)
       real(c_double), intent(in) :: t(*), q(*), u(*), v(*), pmid(*), pint(*), pdel(*), zm(*), zi(*), phis(*), &
                                     pblh(*), tpert(*), landfrac(*), cld(*)
       real(c_double), value :: ztodt
       real(c_double), intent(out) :: ptend_s(*), ptend_q(*), ptend_u(*), ptend_v(*), mcon(*), cme(*), pflx(*), &
                                      zdu(*), rliq(*), rice(*), jctop(*), jcbot(*), prec(*), snow(*), ql(*), rprd(*), &
                                      evapcdp(*), flxprec(*), flxsnow(*), dlf(*), mu(*), md(*), du(*), eu(*), ed(*), &
                                      dp(*), dsubcld(*)
       integer(c_int), intent(out) :: jt(*), maxg(*), ideep(*), lengath(*)
       real(c_double), intent(out) :: cape(*)
     end function zm_conv_tend_batch

     integer(c_int) function zm_conv_tend_batch_gathered(nchunks, ncol, t, q, u, v, pmid, pint, pdel, zm, zi, phis, &
          pblh, tpert, landfrac, cld, ztodt, rliq, rice, jctop, jcbot, prec, snow, cape, dsubcld, jt, maxg, ideep, &
          lengath, pbuf_in_records, rec, rec_cap) bind(C, name='zm_conv_tend_batch_gathered')
       import :: c_int, c_double, c_long_long
       integer(c_int), value :: nchunks
       integer(c_int), intent(in) :: ncol(*)
       real(c_double), intent(in) :: t(*), q(*), u(*), v(*), pmid(*), pint(*), pdel(*), zm(*), zi(*), phis(*), &
                                     pblh(*), tpert(*), landfrac(*), cld(*)
       real(c_double), value :: ztodt
       real(c_double), intent(out) :: rliq(*), rice(*), jctop(*), jcbot(*), prec(*), snow(*), cape(*), dsubcld(*)
       integer(c_int), intent(out) :: jt(*), maxg(*), ideep(*), lengath(*)
       integer(c_int), value :: pbuf_in_records
       real(c_double), intent(out) :: rec(*)
       integer(c_long_long), value :: rec_cap
     end function zm_conv_tend_batch_gathered

     integer(c_int) function zm_conv_tend_2_batch(nchunks, doconvtran, q, pcnst, pdeldry, fracis, ptend_q, ztodt, &
          cnst_is_dry) bind(C, name='zm_conv_tend_2_batch')
       import :: c_int, c_double
       integer(c_int), value :: nchunks
       integer(c_int), intent(in) :: doconvtran(*)
       real(c_double), intent(in) :: q(*)
       integer(c_int), value :: pcnst
       real(c_double), intent(in) :: pdeldry(*), fracis(*)
       real(c_double), intent(inout) :: ptend_q(*)
       real(c_double), value :: ztodt
       integer(c_int), intent(in) :: cnst_is_dry(*)
     end function zm_conv_tend_2_batch

     integer(c_int) function zm_conv_tend_2_batch_gathered(nchunks, lengath, doconvtran, pcnst, cnst_is_dry, q_rec, &
          fracis_rec, pdeldry_rec, dqdt_rec, rec_cap, ztodt) bind(C, name='zm_conv_tend_2_batch_gathered')
       import :: c_int, c_double, c_long_long
       integer(c_int), value :: nchunks
       integer(c_int), intent(in) :: lengath(*), doconvtran(*)
       integer(c_int), value :: pcnst
       integer(c_int), intent(in) :: cnst_is_dry(*)
       real(c_double), intent(in) :: q_rec(*), fracis_rec(*), pdeldry_rec(*)
       real(c_double), intent(out) :: dqdt_rec(*)
       integer(c_long_long), value :: rec_cap
       real(c_double), value :: ztodt
     end function zm_conv_tend_2_batch_gathered

     integer(c_int) function zm_convtran1_fields(pcnst, doconvtran, cnst_is_dry, q, fracis, ptend_q) &
          bind(C, name='zm_convtran1_fields')
       import :: c_int, c_double
       integer(c_int), value :: pcnst
       integer(c_int), intent(in) :: doconvtran(*), cnst_is_dry(*)
       real(c_double), intent(in) :: q(*), fracis(*)
       real(c_double), intent(inout) :: ptend_q(*)
     end function zm_convtran1_fields

     integer(c_int) function zm_org_fields(org, orgt, org2d) bind(C, name='zm_org_fields')
       import :: c_int, c_double
       real(c_double), intent(in)  :: org(*)
       real(c_double), intent(out) :: orgt(*), org2d(*)
     end function zm_org_fields

     integer(c_int) function zm_conv_tend_hist_fields(heat, qtnd, eurt, dif, dnlf, dnif, tend_s, tend_s_snwprd, &
          tend_s_snwevmlt, ntprprd, ntsnprd, seten, pguall, pgdall, icwu, icwd) bind(C, name='zm_conv_tend_hist_fields')
       import :: c_int, c_double
       real(c_double), intent(out) :: heat(*), qtnd(*), eurt(*), dif(*), dnlf(*), dnif(*), tend_s(*), &
                                      tend_s_snwprd(*), tend_s_snwevmlt(*), ntprprd(*), ntsnprd(*), seten(*), &
                                      pguall(*), pgdall(*), icwu(*), icwd(*)
     end function zm_conv_tend_hist_fields

     integer(c_int) function zm_conv_tend_diag_batch(nchunks, ncol, ps, pmid, mu, md, jt, maxg, ideep, lengath, &
          freqzm, mu_out, md_out, pcont, pconb) bind(C, name='zm_conv_tend_diag_batch')
       import :: c_int, c_double
       integer(c_int), value :: nchunks
       integer(c_int), intent(in) :: ncol(*)
       real(c_double), intent(in) :: ps(*), pmid(*)
       ! absent (NULL): taken from the library's device mirror of the last step (gathered mode)
       real(c_double), intent(in), optional :: mu(*), md(*)
       integer(c_int), intent(in), optional :: jt(*), maxg(*), ideep(*), lengath(*)
       real(c_double), intent(out) :: freqzm(*), mu_out(*), md_out(*), pcont(*), pconb(*)
     end function zm_conv_tend_diag_batch

     integer(c_int) function zm_get_timers(n, names, ms) bind(C, name='zm_get_timers')
       import :: c_int, c_ptr, c_float
       integer(c_int), intent(inout) :: n
       type(c_ptr), intent(out) :: names(*)
       real(c_float), intent(out) :: ms(*)
     end function zm_get_timers

     integer(c_int) function zm_set_profiling(on) bind(C, name='zm_set_profiling')
       import :: c_int
       integer(c_int), value :: on
     end function zm_set_profiling

     integer(c_int) function zm_last_error(buf, buflen) bind(C, name='zm_last_error')
       import :: c_int, c_char
       character(kind=c_char), intent(out) :: buf(*)
       integer(c_int), value :: buflen
     end function zm_last_error
  end interface

contains

  !-------------------------------------------------------------------------------
  subroutine zm_batch_init(nchunks, zmconv_org, gathered)
    ! once, after zm_conv_init (zm_convi -> zm_init is done by the shim's zm_convi, zm_conv_intr.F90:376-379);
    ! zmconv_org: the namelist switch zm_convi received (organisation tracer 'ZM_ORG'); gathered: the step returns
    ! the convective columns' records instead of the dense (pcols,pver[p]) arrays (fewer bytes through PCIe and host
    ! memory; INTEGRATION.md section 2 says when to pick it)
    integer, intent(in) :: nchunks
    logical, intent(in), optional :: zmconv_org, gathered
    integer :: m
    nchunks_b = nchunks
    gathered_on = .false.
    if (present(gathered)) gathered_on = gathered
    allocate(ncol_b(nchunks), lengath_b(nchunks))
    allocate(t_b(pcols,pver,nchunks), q_b(pcols,pver,nchunks), u_b(pcols,pver,nchunks), v_b(pcols,pver,nchunks), &
             pmid_b(pcols,pver,nchunks), pdel_b(pcols,pver,nchunks), zm_b(pcols,pver,nchunks), cld_b(pcols,pver,nchunks), &
             pint_b(pcols,pverp,nchunks), zi_b(pcols,pverp,nchunks), phis_b(pcols,nchunks), pblh_b(pcols,nchunks), &
             tpert_b(pcols,nchunks), landfrac_b(pcols,nchunks), ps_b(pcols,nchunks))
    if (gathered_on) then
       rec_len_b = 20*pver + 4                 ! the pbuf fields mu..dp are in the records (pbuf_in_records = 1)
       allocate(rec_b(int(rec_len_b, c_long_long)*pcols*nchunks), rec_base_b(nchunks))
    else
       allocate(ptend_s_b(pcols,pver,nchunks), ptend_q_b(pcols,pver,nchunks), ptend_u_b(pcols,pver,nchunks), &
                ptend_v_b(pcols,pver,nchunks), cme_b(pcols,pver,nchunks), zdu_b(pcols,pver,nchunks), &
                ql_b(pcols,pver,nchunks), rprd_b(pcols,pver,nchunks), evapcdp_b(pcols,pver,nchunks), &
                dlf_b(pcols,pver,nchunks), mu_b(pcols,pver,nchunks), md_b(pcols,pver,nchunks), du_b(pcols,pver,nchunks), &
                eu_b(pcols,pver,nchunks), ed_b(pcols,pver,nchunks), dp_b(pcols,pver,nchunks))
       allocate(mcon_b(pcols,pverp,nchunks), pflx_b(pcols,pverp,nchunks), flxprec_b(pcols,pverp,nchunks), &
                flxsnow_b(pcols,pverp,nchunks))
    end if
    allocate(mu_out_b(pcols,pver,nchunks), md_out_b(pcols,pver,nchunks))
    allocate(rliq_b(pcols,nchunks), rice_b(pcols,nchunks), jctop_b(pcols,nchunks), jcbot_b(pcols,nchunks), &
             prec_b(pcols,nchunks), snow_b(pcols,nchunks), dsubcld_b(pcols,nchunks), cape_b(pcols,nchunks), &
             freqzm_b(pcols,nchunks), pcont_b(pcols,nchunks), pconb_b(pcols,nchunks))
    allocate(jt_b(pcols,nchunks), maxg_b(pcols,nchunks), ideep_b(pcols,nchunks))
    allocate(q3_b(pcols,pver,pcnst,nchunks), fracis_b(pcols,pver,pcnst,nchunks), ptend_q3_b(pcols,pver,pcnst,nchunks), &
             pdeldry_b(pcols,pver,nchunks))
    allocate(heat_b(pcols,pver,nchunks), qtnd_b(pcols,pver,nchunks), eurt_b(pcols,pver,nchunks), dif_b(pcols,pver,nchunks), &
             dnlf_b(pcols,pver,nchunks), dnif_b(pcols,pver,nchunks), tend_s_b(pcols,pver,nchunks), &
             snwprd_b(pcols,pver,nchunks), snwevmlt_b(pcols,pver,nchunks), ntprprd_b(pcols,pver,nchunks), &
             ntsnprd_b(pcols,pver,nchunks), seten_b(pcols,pver,nchunks))
    allocate(pguall_b(pcols,pver,2,nchunks), pgdall_b(pcols,pver,2,nchunks), icwu_b(pcols,pver,2,nchunks), &
             icwd_b(pcols,pver,2,nchunks))
    org_on = .false.
    if (present(zmconv_org)) org_on = zmconv_org
    if (org_on) then
       call cnst_get_ind('ZM_ORG', ixorg)
       allocate(org_b(pcols,pver,nchunks), orgt_b(pcols,pver,nchunks), org2d_b(pcols,pver,nchunks))
    end if
    ! constituent flags: lq(2:) = cnst_is_convtran1(2:) (zm_conv_intr.F90:868), cnst_is_convtran2 (:1009-1010),
    ! cnst_get_type_byind(m) == 'dry' (zm_conv.F90:2087)
    doconvtran1 = 0; doconvtran2 = 0; cnst_is_dry = 0
    do m = 2, pcnst
       if (cnst_is_convtran1(m)) doconvtran1(m) = 1
       if (cnst_is_convtran2(m)) doconvtran2(m) = 1
       if (cnst_get_type_byind(m) == 'dry') cnst_is_dry(m) = 1
    end do
    if (gathered_on) then
       ! convtran2's records: the flagged constituents m = 2..pcnst in ascending order (the library's active list;
       ! doconvtran2(1) is 0)
       nact2 = count(doconvtran2 /= 0)
       allocate(iact2(nact2))
       iact2 = pack([(m, m = 1, pcnst)], doconvtran2 /= 0)
       dry2_any = any(cnst_is_dry(iact2) /= 0)
       allocate(q2rec_b(int(pcols, c_long_long)*nchunks*pver*max(nact2, 1)), &
                fracis2rec_b(int(pcols, c_long_long)*nchunks*pver*max(nact2, 1)), &
                dq2rec_b(int(pcols, c_long_long)*nchunks*pver*max(nact2, 1)))
       if (dry2_any) then
          allocate(pdeldry2rec_b(int(pcols, c_long_long)*nchunks*pver))
       else
          allocate(pdeldry2rec_b(1))
       end if
    end if
  end subroutine zm_batch_init

  !-------------------------------------------------------------------------------
  subroutine zm_batch_gather(ic, state, pblh, tpert, landfrac, cld, fracis)
    ! loop 1 of the split chunk loop: chunk ic's inputs of zm_conv_tend (zm_conv_intr.F90:390-394, 591-600)
    use physics_types, only: physics_state
    integer, intent(in) :: ic
    type(physics_state), intent(in) :: state
    real(r8), intent(in) :: pblh(pcols), tpert(pcols), landfrac(pcols), cld(pcols,pver), fracis(pcols,pver,pcnst)
    ncol_b(ic) = state%ncol
    t_b(:,:,ic) = state%t;       q_b(:,:,ic) = state%q(:,:,1)
    u_b(:,:,ic) = state%u;       v_b(:,:,ic) = state%v
    pmid_b(:,:,ic) = state%pmid; pint_b(:,:,ic) = state%pint; pdel_b(:,:,ic) = state%pdel
    zm_b(:,:,ic) = state%zm;     zi_b(:,:,ic) = state%zi
    phis_b(:,ic) = state%phis;   ps_b(:,ic) = state%ps
    pblh_b(:,ic) = pblh; tpert_b(:,ic) = tpert; landfrac_b(:,ic) = landfrac; cld_b(:,:,ic) = cld
    q3_b(:,:,:,ic) = state%q;    fracis_b(:,:,:,ic) = fracis
    if (org_on) org_b(:,:,ic) = state%q(:,:,ixorg)
  end subroutine zm_batch_gather

  !-------------------------------------------------------------------------------
  subroutine zm_conv_tend_batched(ztodt)
    ! zm_conv_tend for every chunk of the rank (zm_conv_intr.F90:662-886) + its history arithmetic (:685-729)
    real(r8), intent(in) :: ztodt
    integer(c_int) :: rc
    integer :: c
    call t_startf('zm_conv_tend_batch')
    ptend_q3_b = 0._r8                        ! physics_ptend_init(ptend_loc, ..., lq=lq) zeroes the flagged slices
    rc = zm_convtran1_fields(int(pcnst, c_int), doconvtran1, cnst_is_dry, q3_b, fracis_b, ptend_q3_b)
    if (org_on) rc = zm_org_fields(org_b, orgt_b, org2d_b)       ! zm_conv_intr.F90:656-659
    rc = zm_conv_tend_hist_fields(heat_b, qtnd_b, eurt_b, dif_b, dnlf_b, dnif_b, tend_s_b, snwprd_b, snwevmlt_b, &
         ntprprd_b, ntsnprd_b, seten_b, pguall_b, pgdall_b, icwu_b, icwd_b)
    if (gathered_on) then
       rc = zm_conv_tend_batch_gathered(int(nchunks_b, c_int), ncol_b, t_b, q_b, u_b, v_b, pmid_b, pint_b, pdel_b, &
            zm_b, zi_b, phis_b, pblh_b, tpert_b, landfrac_b, cld_b, real(ztodt, c_double), rliq_b, rice_b, jctop_b, &
            jcbot_b, prec_b, snow_b, cape_b, dsubcld_b, jt_b, maxg_b, ideep_b, lengath_b, 1_c_int, rec_b, &
            size(rec_b, kind=c_long_long))
       if (rc /= 0) call zm_batch_abort('zm_conv_tend_batch_gathered', rc)
       rec_base_b(1) = 0
       do c = 2, nchunks_b
          rec_base_b(c) = rec_base_b(c-1) + lengath_b(c-1)
       end do
       ! mu, md, jt, maxg, ideep, lengath from the device mirror the step left
       rc = zm_conv_tend_diag_batch(int(nchunks_b, c_int), ncol_b, ps_b, pmid_b, freqzm=freqzm_b, mu_out=mu_out_b, &
            md_out=md_out_b, pcont=pcont_b, pconb=pconb_b)
    else
       rc = zm_conv_tend_batch(int(nchunks_b, c_int), ncol_b, t_b, q_b, u_b, v_b, pmid_b, pint_b, pdel_b, zm_b, zi_b, &
            phis_b, pblh_b, tpert_b, landfrac_b, cld_b, real(ztodt, c_double), ptend_s_b, ptend_q_b, ptend_u_b, &
            ptend_v_b, mcon_b, cme_b, pflx_b, zdu_b, rliq_b, rice_b, jctop_b, jcbot_b, prec_b, snow_b, ql_b, rprd_b, &
            evapcdp_b, flxprec_b, flxsnow_b, dlf_b, mu_b, md_b, du_b, eu_b, ed_b, dp_b, dsubcld_b, jt_b, maxg_b, &
            ideep_b, lengath_b, cape_b)
       if (rc /= 0) call zm_batch_abort('zm_conv_tend_batch', rc)
       rc = zm_conv_tend_diag_batch(int(nchunks_b, c_int), ncol_b, ps_b, pmid_b, mu_b, md_b, jt_b, maxg_b, ideep_b, &
            lengath_b, freqzm_b, mu_out_b, md_out_b, pcont_b, pconb_b)
    end if
    if (rc /= 0) call zm_batch_abort('zm_conv_tend_diag_batch', rc)
    call t_stopf('zm_conv_tend_batch')
  end subroutine zm_conv_tend_batched

  !-------------------------------------------------------------------------------
  subroutine zm_batch_scatter(ic, lchnk, ptend_all, mcon, cme, pflx, zdu, rliq, rice, jctop, jcbot, &
                              prec, snow, ql, rprd, evapcdp, flxprec, flxsnow, dlf, mconzm, &
                              mu, md, du, eu, ed, dp, dsubcld, jt, maxg, ideep, lengath, &
                              difzm, dnlfzm, dnifzm, dp_cldliq, dp_cldice, org2d)
    ! loop 2 of the split chunk loop: chunk ic's outputs of zm_conv_tend -- ptend_all (lq(1), ls, lu, lv, the
    ! convtran1 constituents and, under zmconv_org, the organisation tracer), the dummy outputs
    ! (zm_conv_intr.F90:390-394), the pbuf fields (:591-621; DIFZM, DNLFZM, DNIFZM, DP_CLDLIQ, DP_CLDICE and
    ! ZM_ORG2D are optional) -- and the history output of :676-857, 882-883
    use physics_types, only: physics_ptend, physics_ptend_init
    integer, intent(in) :: ic, lchnk
    type(physics_ptend), intent(out) :: ptend_all
    real(r8), intent(out) :: mcon(pcols,pverp), cme(pcols,pver), pflx(pcols,pverp), zdu(pcols,pver), rliq(pcols), &
                             rice(pcols), jctop(pcols), jcbot(pcols)
    real(r8), intent(out) :: prec(pcols), snow(pcols), ql(pcols,pver), rprd(pcols,pver), evapcdp(pcols,pver), &
                             flxprec(pcols,pverp), flxsnow(pcols,pverp), dlf(pcols,pver), mconzm(pcols,pverp)
    real(r8), intent(out) :: mu(pcols,pver), md(pcols,pver), du(pcols,pver), eu(pcols,pver), ed(pcols,pver), &
                             dp(pcols,pver), dsubcld(pcols)
    integer,  intent(out) :: jt(pcols), maxg(pcols), ideep(pcols), lengath
    real(r8), intent(out), optional :: difzm(pcols,pver), dnlfzm(pcols,pver), dnifzm(pcols,pver), &
                                       dp_cldliq(pcols,pver), dp_cldice(pcols,pver), org2d(pcols,pver)
    logical  :: lq(pcnst)
    real(r8) :: ftem(pcols,pver)
    integer  :: m, ncol, ixcldliq, ixcldice, i, j
    integer(c_long_long) :: r
    ncol = ncol_b(ic)
    lq(:) = .false.; lq(1) = .true.
    do m = 2, pcnst
       lq(m) = doconvtran1(m) /= 0
    end do
    if (org_on) lq(ixorg) = .true.
    call physics_ptend_init(ptend_all, pcols, 'zm_conv_tend', ls=.true., lu=.true., lv=.true., lq=lq)
    if (gathered_on) then
       ! everything is zero outside the convective columns (rows above lengath for the pbuf fields): zero, then
       ! scatter the chunk's records, column ideep(j) (row j for the pbuf fields) from record rec_base_b(ic)+j
       mcon = 0._r8; cme = 0._r8; pflx = 0._r8; zdu = 0._r8; ql = 0._r8; rprd = 0._r8; evapcdp = 0._r8
       flxprec = 0._r8; flxsnow = 0._r8; dlf = 0._r8
       mu = 0._r8; md = 0._r8; du = 0._r8; eu = 0._r8; ed = 0._r8; dp = 0._r8
       do j = 1, lengath_b(ic)
          r = (rec_base_b(ic) + j - 1) * rec_len_b           ! doubles before the record
          i = ideep_b(j,ic)
          ptend_all%s(i,:)   = rec_b(r+1         : r+pver)
          ptend_all%q(i,:,1) = rec_b(r+pver+1    : r+2*pver)
          ptend_all%u(i,:)   = rec_b(r+2*pver+1  : r+3*pver)
          ptend_all%v(i,:)   = rec_b(r+3*pver+1  : r+4*pver)
          cme(i,:)     = rec_b(r+4*pver+1  : r+5*pver)
          zdu(i,:)     = rec_b(r+5*pver+1  : r+6*pver)
          ql(i,:)      = rec_b(r+6*pver+1  : r+7*pver)
          rprd(i,:)    = rec_b(r+7*pver+1  : r+8*pver)
          evapcdp(i,:) = rec_b(r+8*pver+1  : r+9*pver)
          dlf(i,:)     = rec_b(r+9*pver+1  : r+10*pver)
          mcon(i,:)    = rec_b(r+10*pver+1 : r+11*pver+1)
          pflx(i,:)    = rec_b(r+11*pver+2 : r+12*pver+2)
          flxprec(i,:) = rec_b(r+12*pver+3 : r+13*pver+3)
          flxsnow(i,:) = rec_b(r+13*pver+4 : r+14*pver+4)
          mu(j,:)      = rec_b(r+14*pver+5 : r+15*pver+4)
          md(j,:)      = rec_b(r+15*pver+5 : r+16*pver+4)
          du(j,:)      = rec_b(r+16*pver+5 : r+17*pver+4)
          eu(j,:)      = rec_b(r+17*pver+5 : r+18*pver+4)
          ed(j,:)      = rec_b(r+18*pver+5 : r+19*pver+4)
          dp(j,:)      = rec_b(r+19*pver+5 : r+20*pver+4)
       end do
       mconzm = mcon
    else
       ptend_all%s(:ncol,:) = ptend_s_b(:ncol,:,ic)
       ptend_all%u(:ncol,:) = ptend_u_b(:ncol,:,ic)
       ptend_all%v(:ncol,:) = ptend_v_b(:ncol,:,ic)
       ptend_all%q(:ncol,:,1) = ptend_q_b(:ncol,:,ic)
       mcon = mcon_b(:,:,ic); cme = cme_b(:,:,ic); pflx = pflx_b(:,:,ic); zdu = zdu_b(:,:,ic)
       ql = ql_b(:,:,ic); rprd = rprd_b(:,:,ic); evapcdp = evapcdp_b(:,:,ic)
       flxprec = flxprec_b(:,:,ic); flxsnow = flxsnow_b(:,:,ic); dlf = dlf_b(:,:,ic); mconzm = mcon_b(:,:,ic)
       mu = mu_b(:,:,ic); md = md_b(:,:,ic); du = du_b(:,:,ic); eu = eu_b(:,:,ic); ed = ed_b(:,:,ic); dp = dp_b(:,:,ic)
    end if
    do m = 2, pcnst
       if (lq(m) .and. doconvtran1(m) /= 0) ptend_all%q(:ncol,:,m) = ptend_q3_b(:ncol,:,m,ic)
    end do
    if (org_on) then
       ptend_all%q(:ncol,:,ixorg) = orgt_b(:ncol,:,ic)
       if (present(org2d)) org2d = org2d_b(:,:,ic)
    end if
    ! pbuf fields filled from zm_convr's dif / dnlf / dnif; without zmconv_microp the convective cloud water and ice
    ! are 0 (zm_conv_intr.F90:591-621)
    if (present(difzm))     difzm  = dif_b(:,:,ic)
    if (present(dnlfzm))    dnlfzm = dnlf_b(:,:,ic)
    if (present(dnifzm))    dnifzm = dnif_b(:,:,ic)
    if (present(dp_cldliq)) dp_cldliq = 0._r8
    if (present(dp_cldice)) dp_cldice = 0._r8
    rliq = rliq_b(:,ic); rice = rice_b(:,ic); jctop = jctop_b(:,ic); jcbot = jcbot_b(:,ic)
    prec = prec_b(:,ic); snow = snow_b(:,ic)
    dsubcld = dsubcld_b(:,ic); jt = jt_b(:,ic); maxg = maxg_b(:,ic); ideep = ideep_b(:,ic); lengath = lengath_b(ic)
    ! history (zm_conv_intr.F90:676-729, 796-801, 882-883)
    call outfld('CAPE',     cape_b(:,ic),   pcols, lchnk)
    call outfld('FREQZM  ', freqzm_b(:,ic), pcols, lchnk)
    call outfld('CMFMC_DP', mconzm,         pcols, lchnk)
    call outfld('ZMMU',     mu_out_b(:,:,ic), pcols, lchnk)
    call outfld('ZMMD',     md_out_b(:,:,ic), pcols, lchnk)
    call outfld('DLFZM',    dlf,            pcols, lchnk)
    call outfld('PCONVT  ', pcont_b(:,ic),  pcols, lchnk)
    call outfld('PCONVB  ', pconb_b(:,ic),  pcols, lchnk)
    ftem(:ncol,:) = evapcdp(:ncol,:)
    call outfld('EVAPQZM ', ftem,           pcols, lchnk)
    call outfld('PRECCDZM   ', prec,        pcols, lchnk)
    call outfld('PRECZ   ', prec,           pcols, lchnk)
    if (gathered_on) then                         ! no rank-level ptend_u/v: the chunk's, 0 beyond ncol like the step's
       call outfld('ZMMTU',    ptend_all%u,    pcols, lchnk)
       call outfld('ZMMTV',    ptend_all%v,    pcols, lchnk)
    else
       call outfld('ZMMTU',    ptend_u_b(:,:,ic), pcols, lchnk)
       call outfld('ZMMTV',    ptend_v_b(:,:,ic), pcols, lchnk)
    end if
    call cnst_get_ind('CLDLIQ', ixcldliq)
    call cnst_get_ind('CLDICE', ixcldice)
    call outfld('ZMDICE ', ptend_q3_b(:,:,ixcldice,ic), pcols, lchnk)
    call outfld('ZMDLIQ ', ptend_q3_b(:,:,ixcldliq,ic), pcols, lchnk)
    ! history of zm_convr's, zm_conv_evap's and momtran's intermediates (zm_conv_intr.F90:676-857).  The field names
    ! and the /cpair of each follow the list of the fields this binding used to drop; confirm them against
    ! zm_conv_intr.F90:285-330 (addfld) when the reference source is at hand -- the library returns the procedures'
    ! own quantities, so only this file would change.
    ftem = 0._r8
    ftem(:ncol,:) = heat_b(:ncol,:,ic) / cpair
    call outfld('ZMDT    ', ftem,                 pcols, lchnk)
    call outfld('ZMDQ    ', qtnd_b(:,:,ic),       pcols, lchnk)
    call outfld('EURT    ', eurt_b(:,:,ic),       pcols, lchnk)
    call outfld('DIFZM   ', dif_b(:,:,ic),        pcols, lchnk)
    ftem(:ncol,:) = tend_s_b(:ncol,:,ic) / cpair
    call outfld('EVAPTZM ', ftem,                 pcols, lchnk)
    call outfld('ZMEIHEAT', tend_s_b(:,:,ic),     pcols, lchnk)
    ftem(:ncol,:) = snwprd_b(:ncol,:,ic) / cpair
    call outfld('FZSNTZM ', ftem,                 pcols, lchnk)
    ftem(:ncol,:) = snwevmlt_b(:ncol,:,ic) / cpair
    call outfld('EVSNTZM ', ftem,                 pcols, lchnk)
    call outfld('ZMNTPRPD', ntprprd_b(:,:,ic),    pcols, lchnk)
    call outfld('ZMNTSNPD', ntsnprd_b(:,:,ic),    pcols, lchnk)
    call outfld('ZMFLXPRC', flxprec,              pcols, lchnk)
    call outfld('ZMFLXSNW', flxsnow,              pcols, lchnk)
    if (.not. cam_physpkg_is('cam3')) then       ! momtran is skipped under cam3 (zm_conv_intr.F90:808)
       ftem(:ncol,:) = seten_b(:ncol,:,ic) / cpair
       call outfld('ZMMTT   ', ftem,                 pcols, lchnk)
       call outfld('ZMUPGU  ', pguall_b(:,:,1,ic),   pcols, lchnk)
       call outfld('ZMUPGD  ', pgdall_b(:,:,1,ic),   pcols, lchnk)
       call outfld('ZMVPGU  ', pguall_b(:,:,2,ic),   pcols, lchnk)
       call outfld('ZMVPGD  ', pgdall_b(:,:,2,ic),   pcols, lchnk)
       call outfld('ZMICUU  ', icwu_b(:,:,1,ic),     pcols, lchnk)
       call outfld('ZMICUD  ', icwd_b(:,:,1,ic),     pcols, lchnk)
       call outfld('ZMICVU  ', icwu_b(:,:,2,ic),     pcols, lchnk)
       call outfld('ZMICVD  ', icwd_b(:,:,2,ic),     pcols, lchnk)
    end if
  end subroutine zm_batch_scatter

  !-------------------------------------------------------------------------------
  subroutine zm_batch_gather_2(ic, state, fracis)
    ! inputs of zm_conv_tend_2 (zm_conv_intr.F90:955-1017): state%q, state%pdeldry, fracis; the mass-flux fields
    ! stay in the library's device mirror (pass them as NULL to zm_conv_tend_batch to skip their copy back)
    use physics_types, only: physics_state
    integer, intent(in) :: ic
    type(physics_state), intent(in) :: state
    real(r8), intent(in) :: fracis(pcols,pver,pcnst)
    integer :: n
    integer(c_long_long) :: o, sz
    if (gathered_on) then
       ! the chunk's convective columns ideep(1:n) of the flagged constituents (and their pdeldry), each one section
       n = lengath_b(ic)
       if (n == 0 .or. nact2 == 0) return
       o = int(nact2, c_long_long)*pver*rec_base_b(ic)
       sz = int(n, c_long_long)*pver*nact2
       q2rec_b(o+1:o+sz) = reshape(state%q(ideep_b(1:n,ic),:,iact2), [sz])
       fracis2rec_b(o+1:o+sz) = reshape(fracis(ideep_b(1:n,ic),:,iact2), [sz])
       if (dry2_any) then
          o = int(pver, c_long_long)*rec_base_b(ic)
          pdeldry2rec_b(o+1:o+int(n, c_long_long)*pver) = reshape(state%pdeldry(ideep_b(1:n,ic),:), [n*pver])
       end if
       return
    end if
    q3_b(:,:,:,ic) = state%q
    pdeldry_b(:,:,ic) = state%pdeldry
    fracis_b(:,:,:,ic) = fracis
  end subroutine zm_batch_gather_2

  subroutine zm_conv_tend_2_batched(ztodt)
    real(r8), intent(in) :: ztodt
    integer(c_int) :: rc
    call t_startf('zm_conv_tend_2_batch')
    if (gathered_on) then
       ! mass fluxes, ideep and lengath from the device mirror; lengath_b is checked against it
       rc = zm_conv_tend_2_batch_gathered(int(nchunks_b, c_int), lengath_b, doconvtran2, int(pcnst, c_int), cnst_is_dry, &
            q2rec_b, fracis2rec_b, pdeldry2rec_b, dq2rec_b, size(dq2rec_b, kind=c_long_long), real(ztodt, c_double))
       if (rc /= 0) call zm_batch_abort('zm_conv_tend_2_batch_gathered', rc)
       call t_stopf('zm_conv_tend_2_batch')
       return
    end if
    ptend_q3_b = 0._r8
    rc = zm_conv_tend_2_batch(int(nchunks_b, c_int), doconvtran2, q3_b, int(pcnst, c_int), pdeldry_b, fracis_b, &
                              ptend_q3_b, real(ztodt, c_double), cnst_is_dry)
    if (rc /= 0) call zm_batch_abort('zm_conv_tend_2_batch', rc)
    call t_stopf('zm_conv_tend_2_batch')
  end subroutine zm_conv_tend_2_batched

  subroutine zm_batch_scatter_2(ic, ptend)
    use physics_types, only: physics_ptend, physics_ptend_init
    integer, intent(in) :: ic
    type(physics_ptend), intent(out) :: ptend
    logical :: lq(pcnst)
    integer :: m, ncol, n
    integer(c_long_long) :: o, sz
    ncol = ncol_b(ic)
    do m = 1, pcnst
       lq(m) = doconvtran2(m) /= 0
    end do
    call physics_ptend_init(ptend, pcols, 'convtran2', lq=lq)
    if (gathered_on) then
       ! ptend%q is zero: only the chunk's records go to their columns ideep(1:n) of the flagged constituents
       n = lengath_b(ic)
       if (n == 0 .or. nact2 == 0) return
       o = int(nact2, c_long_long)*pver*rec_base_b(ic)
       sz = int(n, c_long_long)*pver*nact2
       ptend%q(ideep_b(1:n,ic),:,iact2) = reshape(dq2rec_b(o+1:o+sz), [n, pver, nact2])
       return
    end if
    do m = 2, pcnst
       if (lq(m)) ptend%q(:ncol,:,m) = ptend_q3_b(:ncol,:,m,ic)
    end do
  end subroutine zm_batch_scatter_2

  !-------------------------------------------------------------------------------
  subroutine zm_batch_report_timers()
    ! device time of the last profiled step under the reference's GPTL timer names (zm_conv_intr.F90:654-880,
    ! 1019-1025): zm_convr, zm_conv_evap, momtran, convtran1, convtran2 (+ physics_update for the glue kernels)
    integer(c_int) :: n, rc
    type(c_ptr) :: names(8)
    real(c_float) :: ms(8)
    character(kind=c_char), pointer :: cname(:)
    character(len=32) :: name
    integer :: j, i
    n = 8
    rc = zm_get_timers(n, names, ms)
    do j = 1, n
       call c_f_pointer(names(j), cname, [32])
       name = ' '
       do i = 1, 32
          if (cname(i) == c_null_char) exit
          name(i:i) = cname(i)
       end do
       write(iulog,'(a,a,f10.4,a)') ' ZM device timer ', name, ms(j), ' ms'
    end do
  end subroutine zm_batch_report_timers

  !-------------------------------------------------------------------------------
  subroutine zm_batch_abort(what, rc)
    ! the reference's endrun (Brent non-convergence: zm_conv.F90:5401-5410, 5557-5566) with the library's text
    character(len=*), intent(in) :: what
    integer(c_int), intent(in) :: rc
    character(kind=c_char) :: buf(512)
    character(len=512) :: msg
    integer :: i, n
    n = zm_last_error(buf, 512_c_int)
    msg = ' '
    do i = 1, min(n, 511)
       msg(i:i) = buf(i)
    end do
    write(iulog,*) trim(what), ' rc = ', rc, ': ', trim(msg)
    call endrun('**** ZM_CONV '//trim(what)//': '//trim(msg))
  end subroutine zm_batch_abort

end module zm_conv_intr_batched
