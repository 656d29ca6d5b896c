/*
 * vet_b200.h -- C ABI of the B200-native viewport-entropy hot path.
 *
 * The reference (IamArmanNikkhah/viewport-entropy-toolkit) is pure Python and has
 * no FFI of its own; its boundary for this path is the Python API.  Each entry
 * point below names the reference interface it replaces.  Paths are relative to
 * src/viewport_entropy_toolkit/ in the reference:
 *   EU = utilities/entropy_utils.py   DU = utilities/data_utils.py
 *   DT = data_types.py   CFG = config.py
 *   SA = analyzers/spatial_entropy.py   TA = analyzers/transition_entropy.py
 *
 * Conventions
 *   - every function returns a vet_status (0 = ok, negative = error) and never
 *     throws; vet_last_error() returns a thread-local message for the last error;
 *   - the caller owns every buffer; the library owns only the per-configuration
 *     device tables behind the opaque handle (lattices, cell->tile LUTs, FOV weight
 *     tables, scratch) -- one handle per (device, configuration);
 *   - "dev" pointers are device pointers on the handle's device, "host" pointers
 *     are host pointers; `stream` is a cudaStream_t passed as void* (NULL = the
 *     legacy default stream).  Calls taking a stream are asynchronous;
 *   - packed input is [F, U, 3] = (time, 2dmu, 2dmv), frame-major, float32 or
 *     float64 (VET_F32 / VET_F64).  A NaN in 2dmu or 2dmv marks a missing sample
 *     (== a row dropped by dropna at DU:314 / a None cell at SA:131-135);
 *   - tile index outputs use VET_MISSING (0xFFFF) for missing samples;
 *   - data-dependent error conditions that the reference reports by raising
 *     (value outside [0,1]: DU:256-257; frame without users: EU:168-169; frame
 *     pair without a common user: ZeroDivisionError at EU:326) are collected in
 *     a sticky device flag word, read with vet_poll_flags().
 */
#ifndef VET_B200_H
#define VET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vet_handle vet_handle;

typedef enum {
  VET_OK = 0,
  VET_ERR_INVALID_ARG = -1, /* ValueError / ValidationError of CFG:62-67, EU:35-38, DU:236-240 */
  VET_ERR_CUDA = -2,        /* CUDA runtime failure (message in vet_last_error) */
  VET_ERR_UNSUPPORTED = -3, /* configuration outside what the tables can hold */
  VET_ERR_NOMEM = -4
} vet_status;

enum { VET_F32 = 0, VET_F64 = 1 };
enum { VET_TRANSITION_LITERAL = 0, VET_TRANSITION_TEXTBOOK = 1 };
enum { VET_MISSING = 0xFFFF };

/* bits of the sticky flag word (vet_poll_flags) */
enum {
  VET_FLAG_OUT_OF_RANGE = 1,  /* a non-missing 2dmu/2dmv outside [0,1]      (DU:256-257) */
  VET_FLAG_EMPTY_FRAME = 2,   /* a frame with no present user               (EU:168-169) */
  VET_FLAG_NO_COMMON_USER = 4 /* a frame pair without a common user         (EU:326)     */
};

/* AnalyzerConfig (CFG:39-58) + EntropyConfig (EU:20-31), flattened. */
typedef struct {
  int32_t device;                  /* CUDA device ordinal */
  int32_t video_width;             /* CFG:53, must be even (DU:239) */
  int32_t video_height;            /* CFG:54 */
  int32_t num_tile_counts;         /* len(tile_counts), CFG:55 */
  const int32_t* tile_counts;      /* host; tile_count n gives T = 2*int(n/2)+1 tiles (DU:43-45) */
  double fov_angle;                /* EU:29, degrees, 0 < fov <= 360 */
  double power_factor;             /* EU:31, > 0 */
  int32_t use_weight_distribution; /* EU:30 */
  /* Optional host-supplied tables.  NULL => the library derives them itself
   * with libm, following DU:40-54 / DU:283-284,390-397 / DT:204-216.  The
   * Python host passes numpy-made tables so that results follow numpy's
   * arcsin/sin/cos bit for bit (numpy's arcsin differs from libm by 1 ulp on
   * some inputs). */
  const double* const* centres; /* [K] pointers to [T_k,3] lattice centres (generate_fibonacci_lattice, DU:25-56) */
  const double* lon_by_px;      /* [W+1] degrees, after round(.,1) and the wrap quirk (DU:390-395) */
  const double* lat_by_py;      /* [H+1] degrees, after round(.,1) and the wrap quirk (DU:391-397) */
  /* Optional: explicit number of tile centres per tile set, for ARBITRARY tile_centers lists
   * (the reference's free functions accept any List[Vector], EU:70-151,213-219).  When
   * non-NULL, T_k = num_tiles[k] (tile_counts[k] is ignored) and `centres` is required. */
  const int32_t* num_tiles;
  /* Optional: latitude/longitude grid tiling of NaiveSpatialEntropyAnalyzer (NA:39-241,
   * compute_naive_spatial_entropy EU:362-453) instead of the lattice.  When naive_tile_width > 0 the
   * handle has ONE tile set; the "tile" of a sample is the reference's string key
   * "{int((lon+180)/tile_width)}_{int((lat+90)/tile_height)}" (EU:378-381) encoded as
   *     lon_idx * (180/tile_height + 1) + lat_idx          (vet_num_tiles = number of such codes),
   * every sample weighs 1.0 on its tile (EU:357), and use_weight_distribution only selects the
   * normalisation (EU:443-448: by num_tiles = (180/h)*(360/w) when set or when there are more
   * users than tiles, else by the user count).  tile_counts / centres / fov / power are ignored.
   * 360 % tile_width == 0 and 180 % tile_height == 0 are required (EU:414-417). */
  int32_t naive_tile_width;
  int32_t naive_tile_height;
  /* VET_REGIME_AUTO (0): cell tables whenever the video is small enough for them.  VET_REGIME_DIRECT: evaluate
   * every (sample, tile) pair in fp64 without cell tables (the regime of videos too large for the tables; exact,
   * O(users x tiles) per frame) -- what the parity suite compares the table regimes against. */
  int32_t regime;
} vet_config;

enum { VET_REGIME_AUTO = 0, VET_REGIME_DIRECT = 1 };

const char* vet_last_error(void);
const char* vet_version(void);

/* Kernel selection per handle.  The library chooses among its kernels by problem size; an option pins the
 * choice.  Production leaves every option at its default (0 unless stated).  VET_OPT_WEIGHTED_KERNEL is
 * the one a caller may want: the FOV-weighted histogram has two precision modes (see vet_spatial) and results
 * are bit-reproducible across different frame batchings / shardings only when one mode is pinned.  The others exist
 * so that the parity suite can run the kernel generations against each other bit for bit.  The library reads no
 * environment variable. */
#define VET_I8_MIN_FRAMES 384     /* frames per call from which the automatic dispatch takes the tensor-core histogram */
enum {
  VET_OPT_WEIGHTED_KERNEL = 0,   /* 0 auto (tensor cores from VET_I8_MIN_FRAMES frames per call on, where the bound on the entropy error of the
                                    quantised weights holds: DESIGN 4.3), 1 FP64 pipe, 2 tensor cores (int8 slices) */
  VET_OPT_STREAM_KERNEL = 1,     /* 0 auto, 1 plain loads (k_stream_simple), 2 cell histograms only (no direct tile
                                    histograms), 3 global-table regime without the 16-bit privatised histogram */
  VET_OPT_TRANSITION_KERNEL = 2, /* 0 auto (one-pass kernel k_transition4 where its tables fit, the two-pass kernels behind it),
                                    1 k_transition, 2 k_transition2, 3 two-pass kernel k_transition3 alone, one CTA per frame pair */
  VET_OPT_CLUSTER_TAIL = 3,      /* default 1: the pairs the one-pass kernel has left after its full rounds go to its
                                    cluster launch when it pays; 0 never, 2 whenever it can run */
  VET_OPT_T3_PAIR_SCRATCH = 4,   /* 1: keep the 4 B/user pair scratch also when the rows hold tile ids */
  VET_OPT_T3_ASSUME_MISSING = 5, /* 1: always test for missing users (no complete-frame variant) */
  VET_OPT_ANALYZE_OVERLAP = 6,   /* default 1: vet_analyze overlaps its spatial and transition stages; 0 runs them in sequence */
  VET_OPT_HOST_BATCH_FRAMES = 7, /* frames per batch of the host-buffer pipelines; 0 = auto (about 256 MiB of input per batch) */
  VET_OPT_T4_LIST_CAP = 8,       /* one-pass kernel: capacity of the list of users with an unranked tile delta
                                    (0 = 1024; smaller values send more pairs to the two-pass kernels: tests) */
  VET_OPT_CUDA_GRAPH = 9,        /* default 1: vet_spatial / vet_transition / vet_analyze replay their launch sequence as a CUDA
                                    graph from the third identical call on (same buffers, sizes, options, a capturable
                                    stream -- not the legacy default stream); 0: always launch kernel by kernel */
  VET_OPT_HOST_LAYOUT = 10,      /* the *_host entry points read `packed_host` as 0: [F,U,3] = (time, 2dmu, 2dmv) records
                                    (default), 1: [F,U,2] = (2dmu, 2dmv) -- the kernels never read the time column, so a
                                    caller that keeps the frame times itself uploads a third less; the records are widened
                                    on the device */
  VET_OPT_COUNT = 11
};
int vet_set_option(vet_handle* h, int option, int value);
int vet_get_option(const vet_handle* h, int option, int* value);

/* Replaces SpatialEntropyAnalyzer.__init__ / TransitionEntropyAnalyzer.__init__
 * (SA:53-66, TA:53-66): validates the configuration, builds the Fibonacci
 * lattices, the per-cell direction table, the cell->nearest-tile LUT of every
 * tile count (with the brute-force fp64 kernel) and, when weighting is on, the
 * FOV weight tables. */
int vet_create(vet_handle** out, const vet_config* cfg);
int vet_destroy(vet_handle* h);

/* len(generate_fibonacci_lattice(tile_counts[k]))  (DU:43-45). */
int vet_num_tiles(const vet_handle* h, int k);
/* Number of reachable cells (video_height+1)*(video_width+1). */
int64_t vet_num_cells(const vet_handle* h);

/* generate_fibonacci_lattice(tile_counts[k]) -> centres_host[T_k,3]  (DU:25-56). */
int vet_lattice(const vet_handle* h, int k, double* centres_host);
/* Nearest tile of every cell (row-major py*(W+1)+px) for tile count k -> lut_host[cells]. */
int vet_cell_lut(const vet_handle* h, int k, uint16_t* lut_host);

/* Stage 1.  normalize_to_pixel + pixel_to_spherical + round/wrap + Vector.from_spherical
 * (DU:243-286, DU:390-404, DT:183-216) for n samples: packed_dev[n,3] -> vec_dev[n,3]
 * (float64; NaN for missing / out-of-range samples).  cell_dev (optional, may be
 * NULL) receives py*(W+1)+px, or -1 for missing samples. */
int vet_decode(vet_handle* h, const void* packed_dev, int dtype, int64_t n, double* vec_dev,
               int32_t* cell_dev, void* stream);

/* Stage 2.  find_nearest_tile (EU:89-106) for n arbitrary vectors against the
 * lattice of tile count k: vec_dev[n,3] float64 -> idx_dev[n].  fp64 dot of the
 * re-normalised operands (EU:58-61), lowest index among equal maxima (== first
 * minimum of arccos, EU:104). */
int vet_nearest_tile(vet_handle* h, int k, const double* vec_dev, int64_t n, int32_t* idx_dev,
                     void* stream);

/* calculate_tile_weights (EU:108-144) for n arbitrary vectors, dense rows:
 * w_dev[n,T_k] float64 (0 where the reference's dict has no entry). */
int vet_tile_weights(vet_handle* h, int k, const double* vec_dev, int64_t n, double* w_dev,
                     void* stream);

/* find_angular_distances (EU:70-87) for n arbitrary vectors: d_dev[n,T_k] = arccos(clip(dot)),
 * radians (the reference returns [tile_index, distance] pairs; the index is the column). */
int vet_angular_distances(vet_handle* h, int k, const double* vec_dev, int64_t n, double* d_dev,
                          void* stream);

/* vector_angle_distance (EU:41-67) for n independent pairs: d_dev[i] = arccos(clip(dot(a_i/|a_i|, b_i/|b_i|))), radians.
 * Uses the handle only for its device (no tables): one handle serves any number of distinct vectors. */
int vet_vector_angles(vet_handle* h, const double* a_dev, const double* b_dev, int64_t n, double* d_dev,
                      void* stream);

/* compute_spatial_entropy (EU:147-211) for frames of ARBITRARY direction vectors:
 * vec_dev[F,U,3] float64, NaN = absent user.  Same outputs as vet_spatial.  Every
 * (user, tile) pair is evaluated directly (no cell tables); per-tile sums run in user
 * order like EU:190-192.  Also the path vet_spatial takes for videos too large for the
 * cell tables. */
int vet_spatial_vectors(vet_handle* h, const double* vec_dev, int64_t F, int64_t U,
                        double* entropy_dev, double* per_k_dev, double* hist0_dev,
                        uint16_t* assign0_dev, void* stream);

/* compute_transition_entropy (EU:213-332) for frames of arbitrary direction vectors;
 * same outputs as vet_transition. */
int vet_transition_vectors(vet_handle* h, const double* vec_dev, int64_t F, int64_t U,
                           double* entropy_dev, double* per_k_dev, int32_t* prev_count0_dev,
                           uint16_t* pairs0_dev, int mode, void* stream);

/* Stages 1-3 fused.  SpatialEntropyAnalyzer.compute_entropy (SA:107-164) on
 * packed_dev[F,U,3]:
 *   entropy_dev[F]       mean over tile counts of compute_spatial_entropy (EU:147-211)
 *   per_k_dev[K,F]       (optional) entropy per tile count
 *   hist0_dev[F,T_0]     (optional) tile weights of tile_counts[0] (SA:152-154), dense
 *   assign0_dev[F,U]     (optional) nearest tile of tile_counts[0] per user (uint16) */
int vet_spatial(vet_handle* h, const void* packed_dev, int dtype, int64_t F, int64_t U,
                double* entropy_dev, double* per_k_dev, double* hist0_dev, uint16_t* assign0_dev,
                void* stream);

/* Stage 4.  TransitionEntropyAnalyzer.compute_entropy (TA:107-175) on
 * packed_dev[F,U,3]; row r describes frames (r, r+1):
 *   entropy_dev[F-1]        mean over tile counts of compute_transition_entropy (EU:213-332)
 *   per_k_dev[K,F-1]        (optional)
 *   prev_count0_dev[F-1,T_0](optional) users per previous tile, tile_counts[0] (EU:289-292)
 *   pairs0_dev[F-1,U,2]     (optional) (prev,cur) tile per user, tile_counts[0] (EU:276)
 * mode: VET_TRANSITION_LITERAL reproduces the reference's order-dependent
 * bookkeeping (EU:278-318); VET_TRANSITION_TEXTBOOK is an opt-in conditional
 * entropy that the reference does NOT compute. */
int vet_transition(vet_handle* h, const void* packed_dev, int dtype, int64_t F, int64_t U,
                   double* entropy_dev, double* per_k_dev, int32_t* prev_count0_dev,
                   uint16_t* pairs0_dev, int mode, void* stream);

/* Both analyzers in ONE pass over the packed tensor (BASELINE configs[4]: "weighted spatial +
 * transition entropy"): the streaming kernel emits the cell histogram, the tile assignment and the
 * cell ids together, then the spatial epilogue and the transition kernel run on them.  Outputs as in
 * vet_spatial (sp_*, hist0, assign0) and vet_transition (tr_*, prev_count0, pairs0); optional ones may
 * be NULL.  Equivalent to calling vet_spatial and vet_transition, minus one read of the input.
 * The spatial epilogue runs on a stream owned by the handle, forked from and joined back into
 * `stream` with events inside the call: for the caller everything is ordered on `stream`. */
int vet_analyze(vet_handle* h, const void* packed_dev, int dtype, int64_t F, int64_t U,
                double* sp_entropy_dev, double* sp_per_k_dev, double* hist0_dev, uint16_t* assign0_dev,
                double* tr_entropy_dev, double* tr_per_k_dev, int32_t* prev_count0_dev,
                uint16_t* pairs0_dev, int mode, void* stream);

/* Host-buffer variants (the reference-facing call: numpy in, numpy out).  The
 * packed tensor is streamed to the device in frame batches through pinned
 * staging buffers, copies overlapped with the kernels; results are copied
 * back.  Synchronous.  Optional outputs may be NULL. */
int vet_spatial_host(vet_handle* h, const void* packed_host, int dtype, int64_t F, int64_t U,
                     double* entropy_host, double* per_k_host, double* hist0_host,
                     uint16_t* assign0_host);
int vet_transition_host(vet_handle* h, const void* packed_host, int dtype, int64_t F, int64_t U,
                        double* entropy_host, double* per_k_host, int32_t* prev_count0_host,
                        uint16_t* pairs0_host, int mode);
/* vet_analyze on a host tensor: both compute_entropy methods (SA:107-164, TA:107-175) with one upload of the
 * input.  Like vet_transition_host it walks the tensor in frame batches on three streams (upload | kernels |
 * download); the last frame of a batch stays on the device as the first frame of the next one, so no frame is
 * uploaded twice and the device never holds more than two batches (tensors larger than device memory are fine). */
int vet_analyze_host(vet_handle* h, const void* packed_host, int dtype, int64_t F, int64_t U,
                     double* sp_entropy_host, double* sp_per_k_host, double* hist0_host, uint16_t* assign0_host,
                     double* tr_entropy_host, double* tr_per_k_host, int32_t* prev_count0_host,
                     uint16_t* pairs0_host, int mode);

/* Per-viewer exploration entropy: compute_spatial_entropy (EU:147-211) applied to the samples of ONE user over the
 * frames of the video, averaged over the tile counts like SA:142-156 (semantics in vet_users.cuh).  A user without
 * any present sample gets entropy NaN and a zero histogram row (the reference would raise "Empty vector
 * dictionary"); frames without any present user are normal here (no VET_FLAG_EMPTY_FRAME).  Table regimes only:
 * direct-only handles and the latitude/longitude grid tiling return VET_ERR_UNSUPPORTED.
 *
 * acc_dev: [U, S + 1] int64, S = sum_k T_k (tile counts concatenated in k order), column S = present samples.
 * Adds this call's frames into acc (the caller zeroes it once); total_frames >= F fixes the fixed-point scale
 * 2^-b, b = 62 - ceil(log2 total_frames) on weighted handles (0 on unweighted ones: plain counts).  The sums are
 * exact integers, so frames added in any batching, order or over any number of ranks (acc summed across them)
 * give the same bits when every call of one video passes the same total_frames (its global frame count). */
int vet_users_accumulate(vet_handle* h, const void* packed_dev, int dtype, int64_t F, int64_t U,
                         int64_t total_frames, int64_t* acc_dev, void* stream);
/* acc -> entropy_dev[U], per_k_dev[K,U] (optional), hist0_dev[U,T_0] (optional, float64 tile weights of
 * tile_counts[0]); total_frames as in the accumulating calls. */
int vet_users_finish(vet_handle* h, const int64_t* acc_dev, int64_t U, int64_t total_frames,
                     double* entropy_dev, double* per_k_dev, double* hist0_dev, void* stream);

/* Tile transition matrix of a video (semantics in vet_transition_counts.cuh): n_k[p, c] = the (frame pair (f, f+1),
 * user) combinations with the user present in both frames, on tile p of tile count k in frame f and on tile c in
 * frame f+1 -- the pairs of EU:271-276, unweighted -- summed over the frame pairs of the call, and the pooled
 * conditional entropy H_k = -sum (n_pc / N) log2(n_pc / n_p), normalised like the textbook mode (EU:321-327), mean over
 * k.  N = 0, N = 1 and T = 1 give NaN.  A frame pair without a common user raises no flag; out-of-range coordinates set
 * VET_FLAG_OUT_OF_RANGE and count as missing.  Table regimes only: direct-only handles, the latitude/longitude grid
 * tiling and sum_k T_k^2 > 2^28 return VET_ERR_UNSUPPORTED.  Neither call synchronises the stream.
 *
 * acc_dev: int64, the [T_k, T_k] count matrices of all tile counts concatenated in k order (row = previous tile).
 * Adds the (f, f+1) pairs of packed_dev[F,U,3] into acc (the caller zeroes it once).  Batches that overlap by one frame
 * add up to the whole video; the sums are exact integers, so any batching or sharding gives the same bits. */
int vet_transition_counts_accumulate(vet_handle* h, const void* packed_dev, int dtype, int64_t F, int64_t U,
                                     int64_t* acc_dev, void* stream);
/* acc -> entropy_dev[1] (mean over k), per_k_dev[K] (optional), pairs_dev[1] (optional, int64 N).  The row sums go
 * through scratch the handle allocates at creation: finish calls of one handle on different streams must be ordered,
 * like every other call that uses the handle's scratch. */
int vet_transition_counts_finish(vet_handle* h, const int64_t* acc_dev, double* entropy_dev, double* per_k_dev,
                                 int64_t* pairs_dev, void* stream);

/* Per-viewer transition entropy (semantics in vet_user_transitions.cuh): for every user u the conditional entropy of
 * the next tile given the current one over u's own frames -- transition_entropy_textbook (EU:321-327 normalisation) of
 * the (prev_idx, cur_idx) pairs (EU:271-276) of the frames f where u is present in f and f+1, unweighted -- per tile
 * count, and its sequential mean over k (SA:151-156).  One deliberate deviation: a user without a pair (N_u = 0) gets
 * NaN where the textbook mode would raise ZeroDivisionError; N_u = 1 and T = 1 give NaN as in the textbook mode.
 * Out-of-range coordinates set VET_FLAG_OUT_OF_RANGE and count as missing.  A user's outputs are the same bits
 * whatever other users share the call, in any user order, batching or sharding.  Table regimes only: direct-only
 * handles and the latitude/longitude grid tiling return VET_ERR_UNSUPPORTED, and so does F - 1 >= 2^31.  U = 0 or
 * F < 2 is a valid call (every user NaN, 0 pairs).
 *
 * entropy_dev[U]; per_k_dev[K,U] optional; pairs_dev[U] int32 (N_u) optional.  One call = every frame of these U
 * users.  Does not synchronise; after the first call of a size it does not allocate (scratch grown with the handle). */
#define VET_UT_SMEM_RECORDS 3712  /* pair records (runs of one repeated pair) a user's sort keeps in shared memory */
int vet_user_transitions(vet_handle* h, const void* packed_dev, int dtype, int64_t F, int64_t U,
                         double* entropy_dev, double* per_k_dev, int32_t* pairs_dev, void* stream);

/* compute_naive_spatial_entropy (EU:362-453) for frames of ARBITRARY RadialPoints:
 * lonlat_dev[F,U,2] float64 degrees (NaN = absent user, EU:426-427) ->
 *   entropy_dev[F]     normalised entropy (NaN for a frame without users: the reference raises, flag word)
 *   lon_idx_dev[F,U], lat_idx_dev[F,U]   (optional) the two halves of find_naive_tile_index (EU:360-381), -1 = absent
 * Stateless apart from the handle's device and flag word; tile sizes in degrees as in NaiveAnalyzerConfig (CFG:104-105). */
int vet_naive_points(vet_handle* h, const double* lonlat_dev, int64_t F, int64_t U, int32_t tile_width,
                     int32_t tile_height, int32_t use_weight_distribution, double* entropy_dev,
                     int32_t* lon_idx_dev, int32_t* lat_idx_dev, void* stream);

/* Synchronises `stream`, returns the sticky VET_FLAG_* word in *flags and
 * clears it. */
int vet_poll_flags(vet_handle* h, void* stream, uint32_t* flags);

/* Number of kernel launches issued through this handle since creation
 * (bench.py's gpu_launches). */
int64_t vet_launch_count(const vet_handle* h);
/* API calls of this handle that ran as a CUDA graph replay (VET_OPT_CUDA_GRAPH); their kernels are included in
 * vet_launch_count. */
int64_t vet_graph_replays(const vet_handle* h);

/* Per-kernel device timing for the benchmark's roofline line.  When enabled, every
 * launch of the streaming / epilogue / transition / transition-tail / per-viewer transition kernels is bracketed by a CUDA
 * event pair on its own stream (no synchronisation is added).  vet_profile_read
 * waits for the recorded events, returns the summed milliseconds and launch counts
 * per kernel (arrays of VET_KERNEL_COUNT) and clears the record. */
enum {
  VET_KERNEL_STREAM = 0,
  VET_KERNEL_EPILOGUE = 1,
  VET_KERNEL_TRANSITION = 2,
  VET_KERNEL_TRANSITION_TAIL = 3, /* k_transition4<true>: the pairs left after the full rounds, one per CTA cluster;
                                     and k_transition3 over the pairs the one-pass kernel flags */
  VET_KERNEL_USER_ROWS = 4,       /* k_ut_rows of vet_user_transitions */
  VET_KERNEL_USER_ENTROPY = 5,    /* k_ut_entropy of vet_user_transitions */
  VET_KERNEL_COUNT = 6
};
int vet_profile_enable(vet_handle* h, int on);
int vet_profile_read(vet_handle* h, double* ms_by_kernel, int64_t* launches_by_kernel);

#ifdef __cplusplus
}
#endif
#endif /* VET_B200_H */
