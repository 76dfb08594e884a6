/*
 * popsift_b200 -- C ABI of the Blackwell-native SIFT extractor.
 *
 * This is the drop-in boundary for the hot path of alicevision/popsift:
 *     image -> Gaussian pyramid -> DoG extrema -> orientation -> descriptors.
 * The reference has no C ABI; its boundary for this path is the C++ class
 * popsift::Pyramid (reference src/popsift/sift_pyramid.h:88-114:
 * step1 / step2 / get_descriptors / clone_device_descriptors) driven by
 * PopSift::extractDownloadLoop (src/popsift/popsift.cpp:306-344).  Each entry
 * point below names the reference interface it replaces.
 *
 * Conventions: plain pointers and sizes, no C++ types, nothing throws across
 * the ABI.  Functions return 0 (PS_OK) or a negative ps_status; the message
 * is available from ps_last_error().  A context belongs to one CUDA device;
 * its slots are independent in-flight images (one CUDA stream each).
 * There is NO CPU fallback: without a usable CUDA device ps_create fails.
 */
#ifndef POPSIFT_B200_H
#define POPSIFT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PS_ABI_VERSION   3
#define PS_MAX_OCTAVES   20   /* reference sift_conf.h:12  MAX_OCTAVES   */
#define PS_GAUSS_ALIGN   32   /* reference sift_constants.h:37            */
#define PS_GAUSS_LEVELS  12   /* reference sift_constants.h:38            */
#define PS_MAX_ORI       4    /* reference sift_constants.h:54            */
#define PS_MAX_FILTER_GRID 32 /* grid filter: at most 32 x 32 cells        */

typedef enum ps_status {
    PS_OK             =  0,
    PS_ERR_ARG        = -1,  /* bad argument / unsupported configuration        */
    PS_ERR_CUDA       = -2,  /* a CUDA call failed (message in ps_last_error)   */
    PS_ERR_TOO_LARGE  = -3,  /* image exceeds the size the context was made for */
    PS_ERR_STATE      = -4,  /* call order (e.g. download before submit)        */
    PS_ERR_OVERFLOW   = -5   /* more extrema/descriptors than the slot capacity */
} ps_status;

/* enum values follow reference sift_conf.h:33-107 */
enum { PS_MODE_POPSIFT = 0, PS_MODE_OPENCV = 1, PS_MODE_VLFEAT = 2 };
enum { PS_GAUSS_VLFEAT_COMPUTE = 0, PS_GAUSS_VLFEAT_RELATIVE = 1, PS_GAUSS_VLFEAT_RELATIVE_ALL = 2,
       PS_GAUSS_OPENCV_COMPUTE = 3, PS_GAUSS_FIXED9 = 4, PS_GAUSS_FIXED15 = 5 };
enum { PS_DESC_LOOP = 0, PS_DESC_ILOOP = 1, PS_DESC_GRID = 2, PS_DESC_IGRID = 3, PS_DESC_NOTILE = 4 };
enum { PS_NORM_ROOTSIFT = 0, PS_NORM_CLASSIC = 1 };
enum { PS_SCALE_DIRECT = 0, PS_SCALE_DEFAULT = 1 };                                  /* sift_conf.h:75-80   */
enum { PS_FILTER_RANDOM = 0, PS_FILTER_LARGEST_FIRST = 1, PS_FILTER_SMALLEST_FIRST = 2 }; /* sift_conf.h:118-125 */

/* The fields of popsift::Config (reference sift_conf.h:29-409) that the kernels consume. */
typedef struct ps_config {
    int32_t octaves;           /* -1 = auto (popsift.cpp:118-122)                         */
    int32_t levels;            /* 3; clamped to >= 2 (popsift.cpp:86)                      */
    float   sigma;             /* 1.6                                                      */
    float   edge_limit;        /* 10                                                       */
    float   threshold;         /* 0.04 (peak threshold = thr*0.5*255/levels)               */
    float   upscale;           /* 1.0 = -downsampling                                      */
    float   initial_blur;      /* 0.5                                                      */
    int32_t has_initial_blur;  /* 1                                                        */
    int32_t sift_mode;         /* PS_MODE_*                                                */
    int32_t gauss_mode;        /* PS_GAUSS_*  (all six; FIXED9 / FIXED15 need levels == 3 like the reference) */
    int32_t desc_mode;         /* PS_DESC_*   (loop is the fast path; iloop / grid / igrid / notile follow the reference's schemes) */
    int32_t norm_mode;         /* PS_NORM_*                                                */
    int32_t norm_multi;        /* descriptor scaled by 2^norm_multi                        */
    int32_t max_extrema;       /* 100000 per octave                                        */
    /* ABI 2 */
    int32_t scaling_mode;      /* PS_SCALE_*  (DIRECT: level 0 of every octave straight from the input image)         */
    int32_t filter_max_extrema;/* <= 0: grid filter off (reference sift_conf.cu:30, s_orientation.cu:380-383)        */
    int32_t filter_grid_size;  /* 2: cells per image side (s_filtergrid.cu:125)                                      */
    int32_t filter_sort;       /* PS_FILTER_*                                                                        */
} ps_config;

/* Same bytes as popsift::Descriptor (reference sift_extremum.h:69-72). */
typedef struct ps_descriptor { float features[128]; } ps_descriptor;

/* Same bytes as popsift::Feature (reference features.h:23-37), 72 bytes. */
typedef struct ps_feature {
    int32_t        debug_octave;
    float          xpos, ypos, sigma;
    int32_t        num_ori;
    float          orientation[PS_MAX_ORI];
    int32_t        pad_;
    ps_descriptor* desc[PS_MAX_ORI];   /* host pointers into the array given to ps_download */
} ps_feature;

/* Internal extremum record, exposed for tests (octave-local coordinates). */
typedef struct ps_extremum {
    float   xpos, ypos;
    int32_t lpos;
    float   sigma;
    int32_t octave, num_ori, idx_ori;
    float   orientation[PS_MAX_ORI];
} ps_extremum;

typedef struct ps_gauss_tables {
    float   inc_filter[PS_GAUSS_LEVELS * PS_GAUSS_ALIGN];  /* gauss_filter.cu:173-188 */
    float   inc_sigma[PS_GAUSS_LEVELS];
    int32_t inc_span[PS_GAUSS_LEVELS];
    float   dd_filter0[PS_GAUSS_ALIGN];                    /* gauss_filter.cu:227-238, octave 0 */
    float   dd_sigma0;
    int32_t dd_span0;
    float   peak_threshold;                                /* sift_conf.cu:276-279 */
    float   sigma_k;                                       /* sift_constants.cu:27 */
    /* ABI 3: the direct-downscaling rows of every octave (gauss_filter.cu:216-238), used by Config::ScaleDirect:
     * level 0 of octave o is filtered horizontally with row o straight from the input image.  Row 0 == dd_filter0. */
    float   dd_filter[PS_MAX_OCTAVES * PS_GAUSS_ALIGN];
    float   dd_sigma[PS_MAX_OCTAVES];
    int32_t dd_span[PS_MAX_OCTAVES];
    /* the absolute rows of octave 0 (gauss_filter.cu:190-199), used by --gauss-mode vlfeat-direct (VLFeat_Relative_All):
     * every level of octave 0 is filtered straight from the input image with row `level`, horizontally and vertically */
    float   abs_filter[PS_GAUSS_LEVELS * PS_GAUSS_ALIGN];
    float   abs_sigma[PS_GAUSS_LEVELS];
    int32_t abs_span[PS_GAUSS_LEVELS];
    /* the incremental rows transformed for hardware interpolation (gauss_filter.cu:372-405), used by --gauss-mode relative
     * (= vlfeat-hw-interpolated, VLFeat_Relative): [0] centre weight, odd x: fraction u, even x: pair weight v */
    float   inc_ifilter[PS_GAUSS_LEVELS * PS_GAUSS_ALIGN];
    int32_t inc_ispan[PS_GAUSS_LEVELS];
    /* the absolute rows of octaves >= 1 (gauss_filter.cu:200-214): level l straight from level 0 of the same octave; used by
     * --gauss-mode fixed9 / fixed15 */
    float   absn_filter[PS_GAUSS_LEVELS * PS_GAUSS_ALIGN];
    float   absn_sigma[PS_GAUSS_LEVELS];
    int32_t absn_span[PS_GAUSS_LEVELS];
} ps_gauss_tables;

enum { PS_STAGE_H2D = 0, PS_STAGE_PYRAMID = 1, PS_STAGE_EXTREMA = 2, PS_STAGE_ORIENT = 3,
       PS_STAGE_DESC = 4, PS_STAGE_TOTAL = 5, PS_NUM_STAGES = 6 };
enum { PS_PLANE_GAUSS = 0, PS_PLANE_DOG = 1 };

typedef struct ps_ctx ps_ctx;

/* ---- host-only helpers: usable without a GPU -------------------------------------------- */

int  ps_abi_version(void);
/* popsift::Config::Config() defaults (reference sift_conf.cu:18-41) */
void ps_config_default(ps_config* cfg);
/* replaces init_filter + init_constants (reference gauss_filter.cu:127-257, sift_constants.cu:22-53) */
int  ps_gauss_tables_compute(const ps_config* cfg, ps_gauss_tables* out);
/* replaces the printout of Config::setPrintGaussTables() / --print-gauss-tables (gauss_filter.cu:24-121,146-161,247-256): the
 * same text, from this library's tables.  Returns the text length; writes at most cap - 1 characters + 0 into buf (may be NULL) */
int  ps_format_gauss_tables(const ps_config* cfg, char* buf, size_t cap);
/* replaces PopSift::private_apply_scale_factor + Pyramid ctor geometry
 * (reference popsift.cpp:109-126, sift_pyramid.cu:129-134); returns #octaves or <0 */
int  ps_geometry(const ps_config* cfg, int w, int h, int32_t* W, int32_t* H);

/* ---- device path ------------------------------------------------------------------------ */

/* replaces PopSift ctor + Pyramid ctor (reference popsift.cpp:25-48,128-144; sift_pyramid.cu:108-159):
 * allocates n_slots independent pipelines for images up to max_w x max_h on `device`. */
ps_ctx* ps_create(int device, const ps_config* cfg, int max_w, int max_h, int n_slots);
/* replaces Pyramid dtor / PopSift::uninit (reference sift_pyramid.cu:211-225) */
void    ps_destroy(ps_ctx* ctx);
/* last error text; ctx may be NULL for ps_create failures */
const char* ps_last_error(const ps_ctx* ctx);

/* replaces SiftJob::setImg/Image::load + Pyramid::step1 + step2
 * (reference popsift.cpp:293-344,432-437; s_image.cu:69-77; sift_pyramid.cu:227-240):
 * copies the host image to the device and enqueues every kernel of the hot path on the slot's
 * stream.  Returns without waiting for the GPU.
 * Lifetime of `host_img`: a PAGEABLE buffer is copied before the call returns and may be reused or
 * freed at once.  A PAGE-LOCKED buffer (ps_host_alloc, cudaHostAlloc, cudaHostRegister) is read by an
 * asynchronous DMA: it must stay valid and unmodified until ps_wait_input(), ps_counts() or ps_sync()
 * has returned for this slot. */
int ps_submit_u8 (ps_ctx* ctx, int slot, const uint8_t* host_img, int w, int h);
/* float images, value range [0,1) (reference popsift.h:62-69, s_image.cu:262-291) */
int ps_submit_f32(ps_ctx* ctx, int slot, const float* host_img, int w, int h);
/* same, input already resident in device memory of the context's device, `pitch` bytes from one row to the
 * next (pitch >= w, else PS_ERR_ARG); no host copy.  The image is copied device to device on the slot's
 * stream, which is NOT ordered after the caller's streams: the image must be complete when the call is
 * made (synchronize the stream that wrote it first).  `dev_img` is read asynchronously: it must stay valid
 * and unmodified until ps_wait_input(), ps_counts() or ps_sync() has returned for this slot. */
int ps_submit_dev_u8(ps_ctx* ctx, int slot, const uint8_t* dev_img, size_t pitch, int w, int h);

/* replaces Pyramid::readDescCountersFromDevice (reference sift_pyramid.cu:371-379):
 * waits for the slot, returns the number of features and descriptors. */
int ps_counts(ps_ctx* ctx, int slot, int32_t* n_feat, int32_t* n_desc);
/* replaces Pyramid::get_descriptors + prep_features (reference sift_pyramid.cu:250-322):
 * copies n_feat Feature records and n_desc descriptors to the caller's arrays; Feature::desc[]
 * are host pointers into `desc`. */
int ps_download(ps_ctx* ctx, int slot, ps_feature* feat, ps_descriptor* desc);
/* replaces Pyramid::clone_device_descriptors (reference sift_pyramid.cu:324-362), the result path of
 * Config::MatchingMode: copies the slot's n_feat Feature records, n_desc descriptors and the
 * descriptor -> feature reverse map into caller-owned DEVICE arrays (sizes from ps_counts);
 * Feature::desc[] are device pointers into `d_desc`.  Nothing is copied to the host. */
int ps_download_dev(ps_ctx* ctx, int slot, ps_feature* d_feat, ps_descriptor* d_desc, int32_t* d_rev);
/* device memory for ps_download_dev results (thin wrappers of cudaMalloc / cudaFree on the current
 * device) and a blocking device -> host copy for callers without a CUDA toolchain */
void* ps_dev_alloc(size_t bytes);
void  ps_dev_free(void* p);
int   ps_dev_to_host(void* dst_host, const void* src_dev, size_t bytes);
int   ps_host_to_dev(void* dst_dev, const void* src_host, size_t bytes);
/* ordinal of the CUDA device a device pointer belongs to, or -1 */
int   ps_pointer_device(const void* dev_ptr);
/* replaces FeaturesDev::match -> compute_distance (reference features.cu:165-227,282-304): brute-force 2-nearest-
 * neighbour search of every LEFT descriptor among the RIGHT descriptors by squared L2 distance.  d_left / d_right are
 * DEVICE arrays (e.g. the descriptor arrays filled by ps_download_dev); d_out receives n_left x {best index, second
 * index, accept} with accept = (best / second < 0.8f), also in DEVICE memory.  The call returns when the result is
 * complete.  flags: PS_MATCH_AUTO, or force one implementation (PS_MATCH_EXACT: CUDA cores in the reference's
 * evaluation order; PS_MATCH_TENSOR: tcgen05 tf32x3 candidate pass + exact re-rank). */
enum { PS_MATCH_AUTO = 0, PS_MATCH_EXACT = 1, PS_MATCH_TENSOR = 2 };
int ps_match(int device, const ps_descriptor* d_left, int n_left, const ps_descriptor* d_right, int n_right,
             int32_t* d_out, int flags);
/* page-locked host memory for images and results (thin wrappers of cudaHostAlloc / cudaFreeHost).
 * ps_submit_* and ps_download detect page-locked buffers and copy straight from / into them; pageable
 * buffers are staged through the slot's own pinned buffers (one extra host memcpy). */
void* ps_host_alloc(size_t bytes);
void  ps_host_free(void* p);
/* waits until the input image of the slot's last ps_submit_* has been consumed (its copy into the slot's
 * own image buffer is complete): after this a page-locked host buffer or a ps_submit_dev_u8 device buffer
 * may be reused.  Does not wait for the kernels. */
int ps_wait_input(ps_ctx* ctx, int slot);
/* waits for the slot's stream without reading anything */
int ps_sync(ps_ctx* ctx, int slot);

/* replaces Octave::download_and_save_array (reference sift_octave.cu:111-188): one pyramid plane,
 * W*H floats, row-major, no pitch.  which = PS_PLANE_GAUSS (level 0..L+2) / PS_PLANE_DOG (0..L+1). */
int ps_debug_plane(ps_ctx* ctx, int slot, int octave, int level, int which, float* out);
/* extrema of the last image of the slot (after orientation); returns count, fills up to cap */
int ps_debug_extrema(ps_ctx* ctx, int slot, ps_extremum* out, int cap);
/* which evaluation of octave 0 / level 0 is bit-exact for a w x h input scaled to W x H with the reference's `shift`
 * and a row filter of radius R (host arithmetic only, no device needed): 0 = ideal 2x pattern, 1 = neighbouring outputs
 * share their texture fetches, 2 = every tap fetched at its own coordinate (see DESIGN.md, input texture). */
int ps_debug_level0_plan(int w, int h, int W, int H, float shift, int R);
/* geometry of the last image submitted to the slot */
int ps_slot_geometry(ps_ctx* ctx, int slot, int32_t* n_octaves, int32_t* W, int32_t* H);
/* CUDA-event time of each stage of the slot's last image (ms); enable with ps_set_timing(ctx,1) */
int ps_set_timing(ps_ctx* ctx, int enable);
int ps_stage_ms(ps_ctx* ctx, int slot, float ms[PS_NUM_STAGES]);
/* number of kernels this library launched since ps_create (all slots) */
int64_t ps_launch_count(const ps_ctx* ctx);
/* the CUDA stream (cudaStream_t) of a slot, for event timing by the caller */
void* ps_slot_stream(ps_ctx* ctx, int slot);
/* run only the pyramid stage on the slot's current input (benchmark / roofline hook) */
int ps_run_pyramid_only(ps_ctx* ctx, int slot);
/* run ONE pyramid launch on the slot's current planes (roofline hook): level 0 of octave 0 is the
 * input-image kernel, any other (octave, level >= 1) the fused blur+DoG kernel of that level */
int ps_run_level_only(ps_ctx* ctx, int slot, int octave, int level);

#ifdef __cplusplus
}
#endif
#endif /* POPSIFT_B200_H */
