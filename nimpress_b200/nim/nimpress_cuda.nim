## nimpress_cuda.nim -- Nim binding of libnimpress_cuda.so (include/nimpress_cuda.h).
##
## This is the file a nimpress maintainer adds next to src/nimpress.nim.  It could not be compiled
## in the build environment of this repository (no Nim toolchain there); it is a one-to-one
## transcription of the C header, which IS exercised through ctypes and C++ by the test-suite.
##
## Usage inside computePolygenicScores (src/nimpress.nim:592-649): see INTEGRATION.md.

const npcLib* = "libnimpress_cuda.so"

type
  NpcCtx* = distinct pointer

  NpcPolicy* {.bycopy.} = object
    impLocus*: int32      ## ord(ImputeMethodLocus):  ps, homref, fail, ignore
    impMissing*: int32    ## ord(ImputeMethodMissing): homref, ignore
    impSample*: int32     ## ord(ImputeMethodSample): ps, homref, fail, int_ps, int_fail
    reserved*: int32
    mincs*: int64
    maxmis*: float64

  NpcRow* {.bycopy.} = object
    gtRow*: int32         ## row of the genotype slab, -1 when kind != npcKindGt
    eaidx*: int32         ## 0 = REF is the effect allele, k = k-th ALT  (getRawDosages :375-379)
    beta*: float64
    eaf*: float64
    refIsEa*: int32       ## scoreEntry.refseq == scoreEntry.easeq
    kind*: int32          ## npcKind*

  NpcLocus* {.bycopy.} = object
    klass*, used*, eaidx*, reserved*: int32
    ngt*, nmiss*, neff*: int64
    imputed*: float64

const
  npcKindGt* = 0'i32      ## record found and FILTER passes
  npcKindNotCov* = 1'i32  ## not isVariantCovered                         (:526-531)
  npcKindAbsent* = 2'i32  ## findVariant returned nil                     (:536-551)
  npcKindFilter* = 3'i32  ## $variant.FILTER notin [".", "PASS"]          (:553-558)
  npcClassMaxMis* = 4'i32 ## output only: nmissing/n > maxMissingRate     (:565-571)
  npcGtBed* = 0'i32       ## gtWidth of a context over PLINK 1 .bed rows (2 bits per sample, ploidy 2)
  npcGtDose255* = 255'i32 ## gtWidth of a context over BGEN fixed-point dosage rows (uint16 255 x dosage, ploidy 2)
  npcGtDose32* = 32'i32   ## gtWidth of a context over BGEN 32-bit dosage rows (16-byte header with D, uint32 per sample, ploidy 2)
  npcGtPl* = 10'i32       ## gtWidth of a context over FORMAT/PL rows (packed uint32 per sample, ploidy 2)

{.push importc, cdecl, dynlib: npcLib.}
proc npc_create*(ctx: ptr NpcCtx; device: cint; nSamples: int64; ploidy, gtWidth: int32;
                 maxRowsPerBlock: int64; nSlots: int32): cint
proc npc_destroy*(ctx: NpcCtx)
proc npc_last_error*(ctx: NpcCtx): cstring
proc npc_set_stream*(ctx: NpcCtx; cudaStream: pointer): cint
proc npc_set_policy*(ctx: NpcCtx; p: ptr NpcPolicy): cint
proc npc_set_cohort_size*(ctx: NpcCtx; nTotal: int64): cint
proc npc_set_exact_order*(ctx: NpcCtx; on: int32): cint
proc npc_reset*(ctx: NpcCtx): cint
proc npc_stage_acquire*(ctx: NpcCtx; slot: ptr int32; gtHost: ptr pointer; rowStride: ptr int64): cint
proc npc_score_block*(ctx: NpcCtx; slot: int32; nGtRows: int64; rows: ptr NpcRow; nRows: int64): cint
proc npc_score_block_device*(ctx: NpcCtx; gtDev: pointer; rowStride, nGtRows: int64; rows: ptr NpcRow;
                             nRows: int64; rowsOnDevice: int32): cint
proc npc_count_block_device*(ctx: NpcCtx; gtDev: pointer; rowStride, nGtRows: int64; rows: ptr NpcRow;
                             nRows: int64; rowsOnDevice: int32; countsDev: ptr int64): cint
proc npc_accumulate_block_device*(ctx: NpcCtx; gtDev: pointer; rowStride, nGtRows: int64; rows: ptr NpcRow;
                                  nRows: int64; rowsOnDevice: int32; countsDev: ptr int64): cint
proc npc_resident_reserve*(ctx: NpcCtx; capacityRows: int64; grantedRows: ptr int64): cint
proc npc_stage_upload*(ctx: NpcCtx; slot: int32; nGtRows, dstRow: int64): cint
proc npc_resident_adopt*(ctx: NpcCtx; gtDev: pointer; rowStride, nGtRows: int64): cint
proc npc_score_resident*(ctx: NpcCtx; rows: ptr NpcRow; nRows: int64): cint
proc npc_score_resident_multi*(ctx: NpcCtx; nScores: int32; rows: ptr ptr NpcRow; nRows: ptr int64;
                               offsets: ptr float64; scoresOut: ptr ptr float64; nlociOut: ptr int64;
                               lociOut: ptr ptr NpcLocus): cint
proc npc_finish*(ctx: NpcCtx; offset: float64; scoresOut: ptr float64; nlociOut: ptr int64;
                 lociOut: ptr NpcLocus; lociCap: int64; nLociOut: ptr int64): cint
proc npc_partial*(ctx: NpcCtx; sumsOut: ptr float64; nlociOut: ptr int64; lociOut: ptr NpcLocus;
                  lociCap: int64; nLociOut: ptr int64): cint
proc npc_partial_device_ptr*(ctx: NpcCtx; sumsDev: ptr ptr float64; nlociDev: ptr ptr int64): cint
proc npc_normalise*(sums: ptr float64; n, nloci: int64; offset: float64)
proc npc_launch_count*(ctx: NpcCtx): int64
proc npc_multi_contractions*(ctx: NpcCtx): int64
proc npc_kernel_shape*(ctx: NpcCtx; shape: ptr array[8, int32]): cint
proc npc_kernel_shape2*(ctx: NpcCtx; n_rows: int64; shape: ptr array[8, int32]): cint
proc npc_gt_row_bytes*(n_samples: int64; ploidy, gt_width: int32): int64   ## bytes of a row (gt_width npcGtBed: 2-bit rows, npcGtDose255: 2 bytes per sample, npcGtDose32: 16 + 4 per sample, npcGtPl: 4 per sample)
proc npc_pl_weight_table*(out_tab: ptr float64; n: int32): cint   ## T[x] = fl(10^(-x/10)) of FORMAT/PL rows, x = 0 .. n - 1; no device
proc npc_plan_shape*(n_samples: int64; gt_width, num_sms, max_smem: int32; n_rows: int64; exact: int32; plan: ptr array[16, int32]): cint
proc npc_synth_fill_device*(ctx: NpcCtx; gtDev: pointer; rowStride, v0, nRows: int64; seed: uint64;
                            afThr16Dev, missThr24Dev: ptr uint32; altCodeDev: ptr int32): cint
proc npc_version*(): cint
proc npc_warmup*(device: cint): cint
proc npc_create2*(ctx: ptr NpcCtx; device: cint; nSamples: int64; ploidy, gtWidth: int32;
                  maxRowsPerBlock: int64; nSlots: int32; stagingRows: int64): cint
proc npc_create_subset*(ctx: ptr NpcCtx; device: cint; nRowSamples: int64; keep: ptr int64; nKeep: int64; ploidy, gtWidth: int32;
                        maxRowsPerBlock: int64; nSlots: int32; stagingRows: int64): cint
  ## scores keep[0 ..< nKeep] (ascending) of the nRowSamples samples of the staged rows; compacts them on the device
proc npc_gather_rows_device*(ctx: NpcCtx; src: pointer; srcStride, nRows: int64; dst: pointer; dstStride: int64): cint
proc npc_set_keep*(ctx: NpcCtx; keep: ptr int64; nKeep: int64): cint
  ## replaces the keep list of a subset context for rows uploaded after the call (several genotype files)
proc npc_set_dosage_rows*(ctx: NpcCtx; on: int32): cint
proc npc_trace*(ctx: NpcCtx; stamps: ptr array[8, uint64]): cint
# several GPUs: one process (npc_reduce) or one process per GPU over NCCL (npc_comm_*)
proc npc_reduce*(ctxs: ptr NpcCtx; nCtx: int32; offset: ptr float64; scoresOut: ptr float64; nlociOut: ptr int64): cint
proc npc_comm_unique_id*(id128: ptr uint8): cint
proc npc_comm_init*(ctx: NpcCtx; id128: ptr uint8; rank, world: int32): cint
proc npc_comm_combine*(ctx: NpcCtx; offset: ptr float64; scoresOut: ptr float64; nlociOut: ptr int64): cint
proc npc_comm_sum_counts*(ctx: NpcCtx; countsDev: ptr int64; nRows: int64): cint
proc npc_combined_device_ptr*(ctx: NpcCtx; scoresDev: ptr ptr float64; nlociDev: ptr ptr int64): cint
{.pop.}
