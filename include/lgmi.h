/*
 * lgmi.h -- C ABI of liblgmi.so, the B200 (sm_100a) implementation of the
 * L-GIREMI mutual-information step.
 *
 * The reference (gxiaolab/L-GIREMI v0.2.4) is pure Python and has no FFI of
 * its own; the seam this library sits behind is three Python functions:
 *
 *   mismatch_pair_mutual_info(mismatches, min_common_reads)
 *        /root/reference/src/giremi/mutual_information.py:6-45
 *        (called at /root/reference/src/giremi/mismatch.py:389)
 *   mean_mismatch_pair_mutual_info(rows)
 *        /root/reference/src/giremi/mutual_information.py:48-60
 *        (called at /root/reference/src/giremi/mismatch.py:398, after the het
 *         filter at mismatch.py:393-396)
 *   ecdf(x) and its use for `mip` + the threshold call
 *        /root/reference/src/giremi/stat.py:7-29,
 *        /root/reference/src/giremi/script/giremi.py:415-429, :97-114
 *
 * Every entry point below names the reference lines it replaces.  The ctypes
 * binding a reference maintainer would add is shown in INTEGRATION.md and
 * lives in l-giremi_b200/_lib.py.
 *
 * Conventions
 *   - every function returns 0 on success, a negative lgmi_status on error;
 *     lgmi_last_error() gives the message.  No C++ exception crosses the ABI.
 *   - plain pointers + sizes only.  Host buffers passed to *_upload / *_submit
 *     must stay alive until the matching lgmi_batch_sync()/lgmi_wait().
 *   - one lgmi_t per process per GPU (one process per GPU is the scaling
 *     model; there is no collective on this path).  Not thread-safe: callers
 *     serialise calls on one handle.
 *   - there is NO CPU fallback: without a CUDA device lgmi_create() fails.
 */
#ifndef LGMI_H_
#define LGMI_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LGMI_VERSION 100 /* 0.1.0 */

/* the library is built with -fvisibility=hidden; only these are exported */
#if defined(__GNUC__)
#define LGMI_API __attribute__((visibility("default")))
#else
#define LGMI_API
#endif

typedef enum {
  LGMI_OK = 0,
  LGMI_ERR_CUDA = -1,       /* a CUDA runtime call failed                      */
  LGMI_ERR_ARG = -2,        /* bad argument (null, misaligned, out of range)   */
  LGMI_ERR_NOMEM = -3,      /* host or device allocation failed                */
  LGMI_ERR_STATE = -4,      /* call sequence violated (run before upload, ...) */
  LGMI_ERR_NODEVICE = -5,   /* no usable sm_100 device                         */
  LGMI_ERR_UNSUPPORTED = -6 /* shape outside what this build supports          */
} lgmi_status;

/* ----- input encoding ---------------------------------------------------- *
 * A *unit* is one (footprint, strand): the `mismatches[strand]` dict consumed
 * at mutual_information.py:10-26.  It is shipped as three bit-planes per site
 * over the unit's R distinct read names (bit r of word r/32, little endian):
 *     M  read carries the site's major allele   (label 2, :33-38)
 *     m  read carries the site's minor allele   (label 1)
 *     C  read covers the site at all            (label 0 "other" = C & ~M & ~m)
 * Major/minor are decided site-wide by `depth` with the reference's stable
 * tie-break (:25-32); duplicate read names are resolved last-wins (:15-16) by
 * the encoder before packing.  Sites are in ascending position order.
 *
 * Layout of one unit inside the planes buffer (32-bit words):
 *     row(s) = [ M[0..W) | m[0..W) | C[0..W) ],   s = 0..S-1, row stride 3*W
 *     W = row_words = 4*ceil(R/128)   (each plane row is a whole number of
 *                                      16-byte vectors; pad bits are zero)
 * plane_off is the unit's first word, a multiple of 4 (16-byte aligned).
 */
typedef struct {
  uint64_t plane_off; /* first 32-bit word of the unit in the planes buffer    */
  uint32_t n_sites;   /* S >= 0; S < 2 yields no pairs; S <= 65535             */
  uint32_t n_reads;   /* R                                                     */
  uint32_t row_words; /* W = 4*ceil(R/128)                                     */
  uint32_t site_off;  /* first entry of the unit in site_flags / site outputs  */
} lgmi_unit_desc;

/* per-site flag byte */
#define LGMI_SITE_TYPE_MASK 0x03u
#define LGMI_SITE_MISMATCH 0u /* 'mismatch'  (mismatch.py:326-340 typing)      */
#define LGMI_SITE_SNP 1u      /* 'snp'                                         */
#define LGMI_SITE_HET_SNP 2u  /* 'het_snp' -- the only partner type that keeps */
                              /* a pair (mismatch.py:393-396)                  */
#define LGMI_SITE_HAS_OTHER 0x04u /* some read has label 0 at this site; the   */
                                  /* encoder sets it, kernels may also derive  */

/* run modes (bit flags) */
#define LGMI_MODE_ALL_PAIRS 0x0u   /* emit every pair passing min_common       */
                                   /* (= mismatch_pair_mutual_info's return)   */
#define LGMI_MODE_HET_ONLY 0x1u    /* emit only pairs with a het_snp partner   */
                                   /* (= after mismatch.py:393-396); MI is     */
                                   /* still evaluated for every candidate      */
#define LGMI_MODE_EMIT_COUNTS 0x2u /* also emit the 3x3 tables of emitted pairs*/
#define LGMI_MODE_SKIP_NONHET 0x4u /* with HET_ONLY: do not evaluate MI of     */
                                   /* pairs without a het partner (dead work   */
                                   /* in the reference, SURVEY Q7); reported   */
                                   /* separately, never in the headline.  Deep */
                                   /* units with host flags, not pieces, count */
                                   /* only the het sites' rows on the tensor   */
                                   /* cores where that issues at most half the */
                                   /* multiply-adds (lgmi_set_dense_path)      */
#define LGMI_MODE_SPLIT_RECORDS 0x8u /* lgmi_pipeline_step*: deliver the rows as  */
                                   /* two arrays rec_mi / rec_ij (12 bytes per  */
                                   /* row over PCIe instead of 16) and leave    */
                                   /* `records` NULL; the unit of a row follows */
                                   /* from unit_rec_off                         */

#define LGMI_MODE_TIGHT_INPUT 0x20u /* lgmi_pipeline_step_packed: the two-plane     */
                                   /* rows are ceil(R/32) words wide instead of W, */
                                   /* units back to back (no 128-read padding on   */
                                   /* the wire)                                    */
#define LGMI_MODE_COMPACT_OUTPUT 0x40u /* lgmi_pipeline_step*: split rows (as       */
                                   /* SPLIT_RECORDS) with 2-byte (i, j) entries    */
                                   /* when no unit has more than 256 sites, and no */
                                   /* per-site count (site_cnt NULL: it is the     */
                                   /* number of rows a site appears in)            */
#define LGMI_MODE_GRAPH 0x10u       /* lgmi_batch_run: replay the launch chain as   */
                                   /* one CUDA graph (captured on first use per    */
                                   /* (min_common, mode)); the per-kernel times of */
                                   /* lgmi_result are then 0.  Groups of a         */
                                   /* pipelined step always run this way           */
                                   /* (LGMI_GRAPHS=0 in the environment: never)    */

/* one emitted pair == one row [p1,type1,p2,type2,mi] of                       *
 * mutual_information.py:42-44; i<j index the unit's sorted positions.         */
typedef struct {
  uint32_t unit;
  uint16_t i;
  uint16_t j;
  double mi;
} lgmi_pair_rec;

/* results of one batch; pointers are HOST memory owned by the batch, valid    *
 * until the batch is run again or destroyed.                                  */
typedef struct {
  uint64_t n_candidates;        /* sum over units of S(S-1)/2                  */
  uint64_t n_evaluated;         /* candidates whose MI was computed or dropped */
                                /* by the filter: n_candidates, or under       */
                                /* SKIP_NONHET the candidates with a het_snp   */
                                /* partner (counted from the host flag bytes;  */
                                /* n_candidates when the caller filled the     */
                                /* device buffers itself)                      */
  uint64_t n_records;           /* emitted pairs                               */
  const lgmi_pair_rec* records; /* unit order, then pair order (i, then j) --  */
                                /* exactly the reference's row order           */
  const uint32_t* counts;       /* 9 per record [a*3+b], a,b in {0 other,      */
                                /* 1 minor, 2 major}; NULL unless EMIT_COUNTS  */
                                /* (records / counts may also be NULL when     */
                                /* n_records == 0: nothing was allocated)      */
  uint64_t n_sites;             /* length of the two per-site arrays           */
  const double* site_mean;      /* mean MI over het-kept pairs, NaN if none    */
                                /* (mutual_information.py:48-60,               */
                                /*  mismatch.py:476-479)                       */
  const uint32_t* site_cnt;     /* number of het-kept pairs per site           */
  const uint64_t* unit_rec_off; /* n_units+1 offsets of each unit's records    */
  float kernel_ms;              /* device time of all compute kernels of the   */
                                /* run (CUDA events on the launching stream)   */
  float pairs_kernel_ms;        /* device time of the pair kernel alone        */
  float dense_kernel_ms;        /* device time of the tensor-core path         */
                                /* (plane expansion + int8 Gram kernel)        */
  uint32_t n_dense_units;       /* units that took the tensor-core path        */
  uint64_t dense_macs;          /* int8 multiply-accumulates issued for them   */
  float gram_kernel_ms;         /* k_gram_i8 of the last such unit, alone      */
  uint32_t rec_ij_bytes;        /* width of a rec_ij entry: 4, or 2 (see below)*/
  uint64_t gram_macs;           /* multiply-accumulates of that launch         */
  const double* rec_mi;         /* LGMI_MODE_SPLIT_RECORDS: MI of every row    */
  const uint32_t* rec_ij;       /* ... and its i | j << 16; under              */
                                /* LGMI_MODE_COMPACT_OUTPUT with no unit above */
                                /* 256 sites an array of uint16: i | j << 8    */
  uint32_t n_dense_four;        /* of n_dense_units: those whose "other" reads */
                                /* were rare enough for the four-block form    */
                                /* (lgmi_set_dense_path); dense_macs / gram_macs*/
                                /* count the form each unit actually took      */
} lgmi_result;

typedef struct lgmi_ctx lgmi_t;
typedef struct lgmi_batch lgmi_batch_t;

/* ----- context ------------------------------------------------------------ */
LGMI_API int lgmi_version(void);
/* number of CUDA devices this process sees (0: none, or no driver)             */
LGMI_API int lgmi_device_count(void);
/* device: CUDA ordinal.  Fails with LGMI_ERR_NODEVICE if there is no GPU.     */
LGMI_API int lgmi_create(int device, lgmi_t** out);
LGMI_API void lgmi_destroy(lgmi_t* ctx);
LGMI_API const char* lgmi_last_error(const lgmi_t* ctx); /* ctx may be NULL: last create error */
/* Launch on a caller-owned stream (cudaStream_t as void*), e.g. torch's       *
 * current stream so that torch.cuda.Event brackets the kernels. NULL restores *
 * the context's own stream.                                                   */
LGMI_API int lgmi_set_stream(lgmi_t* ctx, void* cuda_stream);
LGMI_API int lgmi_pinned_alloc(lgmi_t* ctx, size_t bytes, void** out);
LGMI_API int lgmi_pinned_free(lgmi_t* ctx, void* ptr);
/* number of kernels this library has launched on the context so far           */
LGMI_API uint64_t lgmi_launch_count(const lgmi_t* ctx);
/* Units with n_sites >= min_sites and n_reads >= min_reads build their        *
 * contingency counts as a dense int8 contraction on the tensor cores          *
 * (tcgen05 / TMEM / TMA) instead of AND+popcount; same counts, bit for bit    *
 * (mutual_information.py:15-40).  Default 48 sites x 8192 reads; applies to   *
 * batches created afterwards.  Tests lower it to force the path.              */
LGMI_API int lgmi_set_dense_threshold(lgmi_t* ctx, uint32_t min_sites, uint32_t min_reads);
/* How the tensor-core path builds the tables (mutual_information.py:24-40: labels *
 * major 2 / minor 1 / other 0).  blocks = 4 (default): while no site of the unit   *
 * has more than max(256, R/64) reads with label "other" -- decided on the device,  *
 * per unit and run -- only the four Gram blocks among {major or minor, major} go   *
 * through the tensor cores and the five cells with an "other" label are counted    *
 * from the listed reads (k_dense_prep, k_other_fix); otherwise, and always with    *
 * blocks = 9, all nine blocks of {covered, major or minor, major}.  Same integers  *
 * either way; applies to batches created afterwards.  Environment                  *
 * LGMI_DENSE_PATH=4/9 sets the default.  Independent of the label form, a run in   *
 * HET_ONLY | SKIP_NONHET on a batch whose flag bytes came from the host computes,  *
 * for every deep unit that is not a piece, only the blocks of the het sites' rows  *
 * against all sites (the het-anchored form) where that issues at most half the    *
 * multiply-accumulates of the pair triangle; dense_macs / gram_macs report the     *
 * form each run took.  lgmi_batch_device_ptrs drops it: the flags are then the     *
 * caller's, unknown to the host.                                                   */
LGMI_API int lgmi_set_dense_path(lgmi_t* ctx, int blocks);
/* Mid-depth units (more than 64 sites or 256 reads, below the dense threshold)   *
 * have their counts built on the tensor cores in one batched launch              *
 * (tensor_cores != 0, default: the warp-specialised k_tile_gram_ws expands the   *
 * bit-planes in the kernel, one tcgen05 int8 MMA per label row block, then       *
 * k_tile_finish) or by tiled AND+popcount (0: k_tile_mi; units deeper than       *
 * 65 535 reads always).  Same integers and the same MI bits either way           *
 * (mutual_information.py:15-41); applies to batches created afterwards.          *
 * Environment LGMI_TILE_PATH=0 selects the popcount form, any other value the    *
 * tensor cores.                                                                  */
LGMI_API int lgmi_set_tile_path(lgmi_t* ctx, int tensor_cores);

/* ----- batched MI step: replaces the per-unit loop                           *
 *   mismatch.py:387-404 = mutual_information.py:6-45 -> het filter -> :48-60  */
/* Builds device-side work tables and sizes the outputs for `units`.           */
LGMI_API int lgmi_batch_create(lgmi_t* ctx, const lgmi_unit_desc* units, uint32_t n_units,
                      uint64_t plane_words, uint64_t n_sites, lgmi_batch_t** out);
LGMI_API void lgmi_batch_destroy(lgmi_batch_t* b);
/* async H2D of planes (plane_words u32) and site_flags (n_sites bytes)        */
LGMI_API int lgmi_batch_upload(lgmi_batch_t* b, const uint32_t* planes, const uint8_t* site_flags);
/* launches the kernels (async).  min_common: keep a pair iff                  *
 * common >= min_common (strict '<' drop, mutual_information.py:19).           */
LGMI_API int lgmi_batch_run(lgmi_batch_t* b, int min_common, uint32_t mode);
/* async D2H of whatever the last run produced, then stream sync; fills *out.  */
LGMI_API int lgmi_batch_download(lgmi_batch_t* b, lgmi_result* out);
/* stream sync only; fills the scalar fields of *out (no record copy)          */
LGMI_API int lgmi_batch_sync(lgmi_batch_t* b, lgmi_result* out);
/* device pointers of the batch's buffers, for device-resident callers         *
 * (benchmarks that generate or keep inputs in HBM).                           */
LGMI_API int lgmi_batch_device_ptrs(lgmi_batch_t* b, void** d_planes, void** d_site_flags,
                           void** d_records, void** d_site_mean);
/* algorithmic bytes of the last run (SURVEY 8d): planes + flags read once,    *
 * 16 B per emitted record, 12 B per site.                                     */
LGMI_API int lgmi_batch_algorithmic_bytes(lgmi_batch_t* b, uint64_t* bytes);

/* ----- split units: one deep unit over several batches / devices ----------- *
 * A unit whose pair work is too large for one device is cut into pieces by    *
 * rows of its pair grid.  The piece of rows [a, b) of a unit of S sites is    *
 * the SUFFIX unit of sites [a, S) (plane_off + 3*a*W, n_sites S - a,          *
 * site_off + a: no re-encoding) with row limit b - a: only its pairs (i, j)   *
 * with i < b - a are evaluated, and they are a prefix of the suffix's pair    *
 * order.  The pieces' records, in row order, with i and j shifted by a, are   *
 * the whole unit's records.                                                   *
 *                                                                             *
 * lgmi_batch_create with a row limit per unit: row_limit[k] == 0 is an        *
 * ordinary unit (exactly as lgmi_batch_create); otherwise unit k is a piece   *
 * and row_limit[k] is a multiple of 128 or n_sites (else LGMI_ERR_ARG).  A    *
 * piece keeps the MI of its pairs in pair order in the batch (NaN: no MI),    *
 * its site_mean / site_cnt entries stay NaN / 0, and n_candidates and         *
 * n_evaluated count its own pairs.                                            */
LGMI_API int lgmi_batch_create_rows(lgmi_t* ctx, const lgmi_unit_desc* units, uint32_t n_units,
                                    const uint32_t* row_limit, uint64_t plane_words, uint64_t n_sites,
                                    lgmi_batch_t** out);
/* async H2D of word_end - word_begin plane words from `planes` (host memory  *
 * holding just those words) to the batch's plane words [word_begin,           *
 * word_end), and of all site_flags (n_sites bytes)                            */
LGMI_API int lgmi_batch_upload_rows(lgmi_batch_t* b, const uint32_t* planes, uint64_t word_begin, uint64_t word_end,
                                    const uint8_t* site_flags);
/* device-to-device copy of n_words plane words of another batch (possibly on  *
 * another device) into this one, queued on dst's stream behind everything     *
 * src's stream has queued at the time of the call (its upload).  Peer access  *
 * is enabled where the devices allow it; the copy works without.             */
LGMI_API int lgmi_batch_copy_planes(lgmi_batch_t* dst, uint64_t dst_word, const lgmi_batch_t* src, uint64_t src_word,
                                    uint64_t n_words);
/* The per-site means and counts of a split unit of n_sites sites: n_pieces    *
 * pieces in row order, piece p being unit unit_in_batch[p] of batches[p],     *
 * each already run (on any device).  Their MI slices are gathered back to     *
 * back on ctx's device and the per-site pass of an unsplit run is applied to  *
 * the result: the same bits as lgmi_batch_create + run of the whole unit      *
 * (mutual_information.py:48-60).  site_flags: the unit's n_sites flag bytes.  *
 * LGMI_ERR_STATE if a piece has not been run, LGMI_ERR_ARG if the pieces do   *
 * not make up the unit.                                                       */
LGMI_API int lgmi_split_means(lgmi_t* ctx, uint32_t n_sites, const uint8_t* site_flags, uint32_t n_pieces,
                              lgmi_batch_t* const* batches, const uint32_t* unit_in_batch, double* mean_out,
                              uint32_t* cnt_out);

/* ----- split units over processes (one process per GPU) -------------------- *
 * The same pieces with their batches in other processes: a piece is exported *
 * as plain bytes (CUDA IPC handles of the batch's plane and dense-MI blocks   *
 * and of an interprocess event), sent by any means, and imported by the       *
 * plane copy and the per-site pass below.  Offsets count from the base of     *
 * each block (a whole device allocation).                                     *
 *                                                                             *
 * Lifetime: an exporting batch must stay alive until every process that      *
 * imported from it has destroyed its importing batch or has returned from     *
 * lgmi_split_means_ipc (a barrier between the processes).                     */
typedef struct {
  uint8_t plane_mem[64];  /* cudaIpcMemHandle_t of the batch's plane block     */
  uint8_t dense_mem[64];  /* cudaIpcMemHandle_t of its dense-MI block          */
  uint8_t event[64];      /* cudaIpcEventHandle_t of its interprocess event,  *
                           * recorded behind all the batch had queued          */
  uint64_t plane_word;    /* the piece's first plane word                      */
  uint64_t plane_words;   /* words of the piece's own rows (3 * W * rows)      */
  uint64_t dense_off;     /* first double of the piece's MI slice              */
  uint64_t dense_pairs;   /* length of that slice: the piece's pairs           */
  uint64_t batch_id;      /* the batch, within the exporting process           */
  uint32_t unit;          /* the piece's unit index in its batch               */
  uint32_t n_sites;       /* sites of the piece's suffix unit                  */
  uint32_t row_limit;     /* its row limit (0: not a piece)                    */
  uint32_t ran;           /* 1 if the batch had been run when this was filled  */
  int32_t pid;            /* exporting process                                 */
  char pci_bus_id[36];    /* the source device, cudaDeviceGetPCIBusId form     */
} lgmi_piece_ipc;         /* 288 bytes                                         */

/* Fills *out for unit `unit` of b (created with a row limit for it) after    *
 * recording b's interprocess event on b's stream, behind everything queued    *
 * so far (the upload, or the run).                                            */
LGMI_API int lgmi_piece_export(lgmi_batch_t* b, uint32_t unit, lgmi_piece_ipc* out);
/* lgmi_batch_copy_planes from a piece exported by another process: n_words   *
 * plane words of its batch from src_word (within the piece's own rows) to     *
 * dst_word of dst, queued on dst's stream behind the piece's event.  The      *
 * source device is found by PCI bus id and must be visible to this process;   *
 * two processes on one device copy device to device.  The mappings opened     *
 * belong to dst (closed by lgmi_batch_destroy; reused by later copies).  A    *
 * piece exported by this process is LGMI_ERR_ARG: use lgmi_batch_copy_planes. */
LGMI_API int lgmi_batch_copy_planes_ipc(lgmi_batch_t* dst, uint64_t dst_word, const lgmi_piece_ipc* src,
                                        uint64_t src_word, uint64_t n_words);
/* lgmi_split_means with pieces in any process, exported after their run      *
 * (else LGMI_ERR_STATE; LGMI_ERR_ARG if they do not make up the unit).  A     *
 * slice from another process is copied behind its piece's event; the          *
 * mappings opened for that are closed before the call returns.  The same     *
 * bits as lgmi_split_means.                                                   */
LGMI_API int lgmi_split_means_ipc(lgmi_t* ctx, uint32_t n_sites, const uint8_t* site_flags, uint32_t n_pieces,
                                  const lgmi_piece_ipc* pieces, double* mean_out, uint32_t* cnt_out);

/* ----- pipelined step over HOST buffers ------------------------------------ *
 * Same result as upload + run + download of one batch (mismatch.py:387-404    *
 * for every unit), but the units are cut into n_chunks consecutive groups of  *
 * about equal work, each on its own stream, so that the H2D copy of group     *
 * k+1, the kernels of group k and the D2H copy of group k-1 overlap.  Units   *
 * must be laid out back to back in `planes` / `site_flags`, in order (what    *
 * the encoder produces); otherwise LGMI_ERR_UNSUPPORTED.  `planes` and        *
 * `site_flags` should be pinned (lgmi_pinned_alloc) for the copies to be      *
 * asynchronous.  Output pointers stay valid until the next step / destroy.    */
typedef struct lgmi_pipeline lgmi_pipeline_t;
LGMI_API int lgmi_pipeline_create(lgmi_t* ctx, const lgmi_unit_desc* units, uint32_t n_units,
                         uint64_t plane_words, uint64_t n_sites, uint32_t n_chunks,
                         lgmi_pipeline_t** out);
LGMI_API int lgmi_pipeline_step(lgmi_pipeline_t* p, const uint32_t* planes, const uint8_t* site_flags,
                       int min_common, uint32_t mode, lgmi_result* out);
/* The same with the input in the packed two-plane form: 2 bits per site and  *
 * read (00 not covered, 01 major, 10 minor, 11 other), row of site s =        *
 * [b0 | b1] with W words each, units back to back (unit k starts at 2/3 of    *
 * its plane_off): a third fewer bytes over PCIe; expanded on the device.      */
LGMI_API int lgmi_pipeline_step_packed(lgmi_pipeline_t* p, const uint32_t* planes2,
                              const uint8_t* site_flags, int min_common, uint32_t mode,
                              lgmi_result* out);
/* The step in two halves, for callers that stream batch after batch (the       *
 * reference's loop over regions, mismatch.py:387-404, taken a batch of regions *
 * at a time): begin queues the uploads and the kernels of every group and      *
 * returns; finish waits for the groups in order, copies the rows back and      *
 * fills *out exactly as lgmi_pipeline_step* does.  With two pipelines on one   *
 * context, begin(B) before finish(A) lets B's uploads share the link with A's  *
 * downloads (the link is full duplex) and keeps kernels queued while the host  *
 * collects A.  collect is the first part of finish on its own: it waits for    *
 * the groups' kernels and queues their downloads without waiting for them, so  *
 * that "begin(k + 2); collect(k + 1); finish(k)" over three pipelines keeps    *
 * both directions of the link queued while the host is inside finish; finish   *
 * collects if nobody has.  The input buffers must stay untouched until finish  *
 * returns; the output arrays of a pipeline are rewritten from its next collect *
 * on.  One step in flight per pipeline: a second begin is LGMI_ERR_STATE, and  *
 * so is a collect or finish without a begin.                                   */
LGMI_API int lgmi_pipeline_begin(lgmi_pipeline_t* p, const uint32_t* planes, const uint8_t* site_flags,
                        int min_common, uint32_t mode);
LGMI_API int lgmi_pipeline_begin_packed(lgmi_pipeline_t* p, const uint32_t* planes2,
                               const uint8_t* site_flags, int min_common, uint32_t mode);
LGMI_API int lgmi_pipeline_collect(lgmi_pipeline_t* p);
LGMI_API int lgmi_pipeline_finish(lgmi_pipeline_t* p, lgmi_result* out);
LGMI_API void lgmi_pipeline_destroy(lgmi_pipeline_t* p);

/* one-shot convenience: create + upload + run + download (+ destroy on wait)  */
LGMI_API int lgmi_submit(lgmi_t* ctx, const lgmi_unit_desc* units, uint32_t n_units,
                const uint32_t* planes, uint64_t plane_words,
                const uint8_t* site_flags, uint64_t n_sites, int min_common,
                uint32_t mode);
LGMI_API int lgmi_wait(lgmi_t* ctx, lgmi_result* out); /* result valid until next submit */

/* ----- mean of pre-computed rows: mutual_information.py:48-60 -------------- *
 * CSR form: site s owns values[offsets[s] .. offsets[s+1]) in row order.      *
 * mean[s] = sum/len with CPython's compensated float sum; NaN for empty.      */
LGMI_API int lgmi_site_mean_csr(lgmi_t* ctx, const uint64_t* offsets, const double* values,
                       uint64_t n_sites, double* mean_out);

/* ----- global pass: stat.py:7-29 + giremi.py:415-429 + :97-114 ------------- *
 * mip[s]  = NaN if mean[s] is NaN, else (#het means strictly below mean[s])   *
 *           mapped through y = [0] ++ linspace(1/n, 1, n)                     *
 * call[s] = 1 if mean notna & mip<=thr & type==mismatch                       *
 *           2 if mean notna & mip> thr & type!=mismatch, else 0               *
 * site_flags carries the type in its low 2 bits.  call may be NULL.           */
LGMI_API int lgmi_ecdf(lgmi_t* ctx, const double* mean, const uint8_t* site_flags, uint64_t n,
              double threshold, double* mip, uint8_t* call);
/* ecdf(x)(samples): y[searchsorted(sort(x), samples, 'left')]  (stat.py:16-27)*
 * NaNs in x sort last and a NaN sample lands on the first of them, as numpy    *
 * orders them.                                                                 */
LGMI_API int lgmi_ecdf_eval(lgmi_t* ctx, const double* x, uint64_t n, const double* samples,
                   uint64_t n_samples, double* out);
/* ecdf(x) itself (stat.py:16-19), built ONCE: sorted_out = sort(x) (n values)  *
 * and y_out = [0] ++ linspace(1/n, 1, n) (n + 1 values), both computed on the  *
 * device.  The callable the reference returns (stat.py:21-27) is then          *
 * y_out[searchsorted(sorted_out, sample, 'left')]: the CLI applies it row by   *
 * row (giremi.py:424-428), which must not cost a device round trip per row.    */
LGMI_API int lgmi_ecdf_table(lgmi_t* ctx, const double* x, uint64_t n, double* sorted_out, double* y_out);

/* ----- site x splice-site MI: calculate_site_splice_mi.py:106-125 ---------- *
 * The reference's second mutual_info_score call site, for the requested       *
 * (site, allele, splice site) triples only.  Synchronous.                     *
 *   entries  site s owns entries [entry_off[s], entry_off[s+1]): one per list *
 *            entry of the site (a read listed twice counts twice), its read   *
 *            entry_read[p] < n_reads and the index entry_allele[p] of the     *
 *            allele list it comes from, numbered within the site.  At most   *
 *            64 distinct alleles per site (index >= 64: UNSUPPORTED).         *
 *   splices  read r has splice sites splice_id[splice_off[r] ..              *
 *            splice_off[r+1]), ascending and unique (membership is a set).    *
 *   triples  tri_site[t] < n_sites, tri_allele[t] (an allele index of the     *
 *            site), tri_splice[t] (any id; one no read has gives 0.0).        *
 * Over the N entries of the site: x entries whose read is in the allele's     *
 * list at the site (by read, :121), y whose read has the splice site (:122),  *
 * xy both.  table_out (optional, 4 per triple) receives [N-x-y+xy, y-xy,      *
 * x-xy, xy] (rows "with seq", columns "with splice"), mi_out[t] its MI (:123; *
 * 0.0 for one class).  LGMI_ERR_ARG for a NULL array, an offset array that   *
 * does not start at 0 or decreases, an id out of range or splice ids out of   *
 * order.                                                                      */
LGMI_API int lgmi_site_splice_mi(lgmi_t* ctx, uint32_t n_sites, const uint64_t* entry_off,
                                 const uint32_t* entry_read, const uint32_t* entry_allele, uint32_t n_reads,
                                 const uint64_t* splice_off, const uint32_t* splice_id, uint64_t n_triples,
                                 const uint32_t* tri_site, const uint32_t* tri_allele, const uint32_t* tri_splice,
                                 double* mi_out, uint32_t* table_out);

/* ----- host-side native pieces either side of the step (no device needed) --- *
 * One read's short-form cs tag (minimap2 --cs): its substitutions in contig    *
 * coordinates (0-based) with the splice-distance filter applied, and its       *
 * introns.  Replaces, per read, CS.from_cs_tag_string + get_mismatches +       *
 * get_introns (giremi/cs.py:8-41, :573-613) and FILTER 1 of                    *
 * giremi/mismatch.py:99-141 (merged +-min_dist intervals around every intron   *
 * start and end, membership start <= pos < end as in utils.py:4-31).           *
 * mm_ref / mm_alt are upper-case bases.  Returns LGMI_ERR_ARG for a mark the   *
 * reference does not know, LGMI_ERR_NOMEM (counts still set) when a capacity   *
 * is too small.                                                                */
LGMI_API int lgmi_cs_scan(const char* cs, uint64_t cs_len, int64_t ref_start, int min_dist_from_splice,
                 uint32_t cap_mismatch, int64_t* mm_pos, char* mm_ref, char* mm_alt,
                 uint32_t* n_mismatch, uint32_t cap_intron, int64_t* intron_lo, int64_t* intron_hi,
                 uint32_t* n_intron);
/* One unit from its flattened `mismatches[strand]` dict to bit-planes + flag   *
 * bytes (the layout above), with the dict semantics the kernels cannot see:    *
 * a read listed twice at a site keeps its last allele                          *
 * (mutual_information.py:15-16), major / minor by `depth` descending with the  *
 * stable tie-break (:25-32), every other allele -> "other" (:33-38).           *
 * Sites in ascending position order.  Per site s: n_depth_entries[s] pairs     *
 * (depth_allele, depth_value) in the depth dict's order, n_nt_entries[s] pairs *
 * (nt_allele, nt_n_names) in the nt dict's order; allele ids are any integers  *
 * consistent within a site; the read names of all lists, in order, are one     *
 * newline-separated blob.  Outputs: planes (3 * n_sites * W words, W returned  *
 * in row_words_out), site_flags, bad_site (1: fewer than two alleles in        *
 * `depth`), the number of distinct reads.  LGMI_ERR_NOMEM if plane_cap_words   *
 * is too small (n_reads_out / row_words_out are set: call again).              */
LGMI_API int lgmi_encode_unit(uint32_t n_sites, const uint8_t* site_type, const uint32_t* n_depth_entries,
                     const uint32_t* depth_allele, const int64_t* depth_value,
                     const uint32_t* n_nt_entries, const uint32_t* nt_allele,
                     const uint32_t* nt_n_names, const char* names_blob, uint64_t blob_len,
                     uint64_t plane_cap_words, uint32_t* planes, uint8_t* site_flags,
                     uint8_t* bad_site, uint32_t* n_reads_out, uint32_t* row_words_out);

/* ----- multi-GPU partitioning (no collective; SURVEY 8e) ------------------- *
 * cost(unit) = S(S-1)/2 * ceil(R/64).  Longest-processing-time greedy into    *
 * n_bins; bin_of[u] receives the bin.  Deterministic (ties: lower index).     */
LGMI_API uint64_t lgmi_unit_cost(uint32_t n_sites, uint32_t n_reads);
LGMI_API int lgmi_partition_lpt(const uint64_t* cost, uint32_t n_units, uint32_t n_bins,
                       uint32_t* bin_of, uint64_t* bin_load);

#ifdef __cplusplus
}
#endif
#endif /* LGMI_H_ */
