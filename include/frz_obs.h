/*
 * frz_obs.h -- compact observation download of libfrz.so (additive to the C ABI of frz.h).
 *
 * A policy that runs on the host reads the observations of every step, and the link between host and device is the
 * slowest hop of such a step.  Most observation values are small integers stored wide (int32 task rows whose values
 * fit a byte, one byte per 0/1 mask entry, configuration constants repeated per environment), so this download
 * encodes them on the device into a compact format, in device staging buffers, and then moves exactly the live bytes
 * into the caller's page-locked host buffers (device-mapped under unified addressing) with 16-byte stores: the live
 * sizes are read on the device, so no host read sits between the encoding and the transfer.
 *
 * The library knows array descriptors only, never domains; which array is narrowed to which type is decided once by
 * the caller from bounds its configuration guarantees (free_range_zoo_b200/utils/compact.py).
 *
 * Layout of the download for B environments with counts[b] live rows each:
 *  - offsets[0 .. B]: exclusive prefix sum of counts (int32).  Counts outside [0, smallest capacity of the ROWS and
 *    MASK_BITS arrays] are clamped to it and set the overflow flag.
 *  - DENSE array: src = [B, capacity rows, src_columns]; dst = [B, capacity, columns] holds columns
 *    [column_first, column_first + columns) of every row, converted to dst_type.
 *  - ROWS array: src = [B, groups, capacity rows, src_columns] of which rows 0 .. counts[b]-1 of every block are live;
 *    in dst, environment b's block g starts at row offsets[b] * groups + g * counts[b] (rows of `columns` elements of
 *    dst_type) -- the packing of frz_gather_live_rows, narrowed.
 *  - MASK_BITS array: src = uint8 [B, groups, capacity]; environment b's bits start on byte
 *    mask_offsets[b] = sum over b' < b of ceil(groups * counts[b'] / 8), and bit g * counts[b] + t (LSB first) is
 *    src[b, g, t] != 0.  The layout depends on the counts alone, never on how a batch is cut.
 *  - A value that does not fit its dst_type sets the overflow flag (status[0]) to 1 (the configuration bound the type was chosen from
 *    was violated, e.g. by an initial state from outside the configuration); the caller must not use the download.
 */
#ifndef FRZ_OBS_H_
#define FRZ_OBS_H_

#include "frz.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef enum { FRZ_OBS_DENSE = 0, FRZ_OBS_ROWS = 1, FRZ_OBS_MASK_BITS = 2 } FrzObsKind;

/* element types: sources are int32, float32 or uint8; int32 sources narrow to int16 / int8 / uint8 */
typedef enum { FRZ_OBS_I32 = 0, FRZ_OBS_I16 = 1, FRZ_OBS_I8 = 2, FRZ_OBS_U8 = 3, FRZ_OBS_F32 = 4 } FrzObsType;

typedef struct {
  const void* src;        /* device */
  void* dst;              /* device staging of the encoding, room for the whole padded array in dst_type */
  void* host;             /* page-locked host memory of the same size that receives the live bytes; NULL = leave the
                             encoding in dst (the caller downloads it) */
  int32_t kind;           /* FrzObsKind */
  int32_t src_type;       /* FrzObsType of src */
  int32_t dst_type;       /* FrzObsType of dst (MASK_BITS: FRZ_OBS_U8) */
  int32_t groups;         /* row blocks per environment (DENSE: 1) */
  int32_t capacity;       /* padded rows per (environment, block) in src */
  int32_t src_columns;    /* elements per src row (MASK_BITS: 1) */
  int32_t column_first;   /* first src column copied */
  int32_t columns;        /* columns copied per row */
} FrzObsArray;

typedef struct {
  const int32_t* counts;  /* device [B]: live rows per environment */
  int32_t* offsets;       /* device [B + 1] */
  int32_t* host_offsets;  /* page-locked host [B + 1] that receives offsets, or NULL */
  int32_t* scan;          /* device scratch int32 [2 * (B + 1)]: (row offset, mask byte offset) per environment */
  int32_t* scratch;       /* device scratch int32 [2 * ((B + 1023) / 1024 + 1)] */
  uint32_t* status;       /* page-locked host [4]: overflow flag (1 when a value did not fit its dst_type), live rows
                             (offsets[B]), mask bytes (mask_offsets[B]), 0 -- the sizes a reader needs, without a scan */
  const FrzObsArray* arrays;
  int32_t array_count;
  int32_t mask_groups;    /* groups of every MASK_BITS array (mask bits per live row) */
} FrzObsDownload;

/* Encode the observations of all `parallel_envs` environments into the compact format and move the live bytes into
 * the page-locked host buffers of `download`.  Every host pointer is resolved with cudaHostGetDevicePointer first:
 * memory that is not page-locked host memory mapped for the current device is refused with FRZ_ERR_UNSUPPORTED before
 * anything is launched.  dst, host, offsets and host_offsets must be 16-byte aligned.  Only enqueues work on `stream`;
 * the host buffers are complete once the stream has been synchronised. */
int frz_observe_compact(const FrzObsDownload* download, int32_t parallel_envs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FRZ_OBS_H_ */
