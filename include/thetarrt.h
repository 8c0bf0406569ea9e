/*
 * thetarrt.h -- C ABI of libthetarrt.so, the B200 (sm_100a) implementation of
 * theta-rrt's data-parallel planning inner loop.
 *
 * The reference (eshira/theta-rrt) is pure Python and has no FFI; the boundary
 * a maintainer would bind is the set of Python callables below.  Each entry
 * point names the reference interface it replaces (file:line into the
 * reference tree).  INTEGRATION.md shows the ctypes stubs.
 *
 * Conventions
 *   - every pointer prefixed d_ is a DEVICE pointer owned by the caller
 *     (PyTorch tensors in the Python shim); the library never allocates or
 *     frees device memory and keeps no global state;
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work on
 *     it and never synchronise;
 *   - return value: trrt_error (0 = ok).  No exceptions cross the ABI;
 *   - per-query results that the reference reports through None/False/raised
 *     exceptions come back as trrt_status codes in an output array.
 *   - maps must be square (H == W): the reference's own bounds test compares x
 *     with shape[0] and y with shape[1] (search.py:21) and indexes
 *     imarray[y][x] (search.py:30), which is only self-consistent for square
 *     images; non-square input returns TRRT_ERR_NONSQUARE_MAP.
 */
#ifndef THETARRT_H
#define THETARRT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRRT_VERSION 200 /* 0.2.0 */

/* Parameters the reference keeps in `builtins` (main.py:15-32). */
typedef struct trrt_params {
    int32_t thetastar;      /* builtins.THETASTAR       main.py:15 */
    int32_t forwardonly;    /* builtins.FORWARDONLY     main.py:19 */
    double bikelength;      /* builtins.bikelength      main.py:18 */
    double leftconstraint;  /* builtins.LEFTCONSTRAINT  main.py:20 */
    double rightconstraint; /* builtins.RIGHTCONSTRAINT main.py:21 */
    double frontclearance;  /* builtins.frontclearance  main.py:22 */
    double maxdrivedist;    /* builtins.maxdrivedist    main.py:27 */
    double tol_xy;          /* builtins.tol_xy          main.py:28 */
    double tol_ang;         /* builtins.tol_ang         main.py:29 */
    double weightxy;        /* builtins.weightxy        main.py:30 */
} trrt_params;

typedef enum trrt_error {
    TRRT_OK = 0,
    TRRT_ERR_INVALID_ARGUMENT = 1,
    TRRT_ERR_NONSQUARE_MAP = 2,
    TRRT_ERR_MAP_TOO_LARGE = 3, /* side > 32768 */
    TRRT_ERR_WORKSPACE_TOO_SMALL = 4,
    TRRT_ERR_CUDA = 5,
    TRRT_ERR_NO_DEVICE = 6
} trrt_error;

/* per-query status (reference behaviour in brackets) */
typedef enum trrt_status {
    TRRT_OK_FOUND = 0,                    /* [path list / sol is a node]                       */
    TRRT_OK_NOT_FOUND = 1,                /* [astar -> False, search.py:307; rrt sol=None]     */
    TRRT_ERR_ENDPOINT_INVALID = 2,        /* [astar prints + False, search.py:222-224]         */
    TRRT_ERR_ENDPOINT_BLOCKED = 3,        /* [astar prints + False, search.py:225-227]         */
    TRRT_ERR_REF_RAISES_DRIVE_NONE = 4,   /* [TypeError: drive() after straight steer, rrt.py:170-171,275] */
    TRRT_ERR_REF_RAISES_ARGMIN_EMPTY = 5, /* [ValueError: np.argmin([]), search.py:262]        */
    TRRT_ERR_CAPACITY = 6,                /* heap / path / node capacity of the call exceeded  */
    TRRT_ERR_REF_RAISES_NO_NEAREST = 7    /* [TypeError: findnearest of a childless tree, main.py:79-81] */
} trrt_status;

/* outcome of one RRT loop iteration (rrt.py:141-201) */
typedef enum trrt_iter_code {
    TRRT_IT_NEW_NODE = 0,         /* rrt.py:179-180 vertex inserted                 */
    TRRT_IT_EXISTING_NODE = 1,    /* qnew already a key of G: edge appended only    */
    TRRT_IT_QRAND_BLOCKED = 2,    /* rrt.py:148                                     */
    TRRT_IT_QRAND_IN_TREE = 3,    /* rrt.py:151                                     */
    TRRT_IT_STEER_CONSTRAINT = 4, /* rrt.py:166                                     */
    TRRT_IT_ARC_BLOCKED = 5,      /* rrt.py:174                                     */
    TRRT_IT_NOT_RUN = 255
} trrt_iter_code;

int trrt_version(void);
const char *trrt_error_string(int err);
/* last CUDA error string seen by this thread's most recent failing call ("" if none) */
const char *trrt_last_cuda_error(void);
void trrt_default_params(trrt_params *p); /* main.py:15-32 defaults */

/* ---------------------------------------------------------------------------
 * Occupancy grid.  Replaces builtins.imarray (main.py:38-42) + search.valid /
 * search.freespace (search.py:17-33).
 * Packed layout: n_maps maps, each H rows of wpr = (W+31)/32 uint32 words;
 * pixel (x, y) is bit (x & 31) of word [y*wpr + (x >> 5)], 1 = free.  Padding
 * bits are 0 (blocked).  d_free is the byte image [n_maps][H][W], non-zero =
 * free, exactly np.array(Image.open(p).convert('1')).
 * ------------------------------------------------------------------------- */
size_t trrt_grid_words(int H, int W);
int trrt_pack_grid(const uint8_t *d_free, int n_maps, int H, int W, uint32_t *d_bits, void *stream);

/* ---------------------------------------------------------------------------
 * K4 los_batch.  Replaces search.lineofsight (search.py:35-41) incl. bresenham
 * / plotLineLow / plotLineHigh (search.py:43-94) for n independent segments.
 * d_seg: int32 [n][4] = (x0, y0, x1, y1) already int()-truncated.
 * d_map_id: int32 [n] map index per segment, or NULL (all map 0).
 * d_out: uint8 [n], 1 = line of sight.
 * ------------------------------------------------------------------------- */
int trrt_los_batch(const uint32_t *d_bits, int n_maps, int H, int W, const int32_t *d_map_id, const int32_t *d_seg,
                   int64_t n, uint8_t *d_out, void *stream);

/* ---------------------------------------------------------------------------
 * K4b los_batch_tiled.  Same contract and results as trrt_los_batch
 * (search.lineofsight, search.py:35-94), over a second copy of the grid laid
 * out so that the 8 pixels of a ray inside one aligned block of 8 along its
 * driving axis come from ONE 16-byte load, for rays of any direction.
 * Layout per map, tp = (side+7)/8: [orientation 2][K tp+1][c tp] entries of
 * 16 bytes; in orientation 0 (rays driven by x, plotLineLow search.py:58-75)
 * byte j bit i of entry (K, c) is pixel (x = 8c+i, y = 8K-8+j), in
 * orientation 1 (driven by y, plotLineHigh search.py:77-94) pixel
 * (x = 8K-8+j, y = 8c+i); 1 = free, outside the image 0.  Entries overlap by
 * half so that the 8x8 window a block can touch is always inside one entry.
 * trrt_tile_grid derives the copy from the packed rows of trrt_pack_grid;
 * d_tiles must be 16-byte aligned.  Lanes take the next segment as soon as
 * theirs is decided, so long and short rays can be mixed freely.
 * ------------------------------------------------------------------------- */
size_t trrt_tile_words(int H, int W); /* uint64 words per map = 4 * (tp+1) * tp */
int trrt_tile_grid(const uint32_t *d_bits, int n_maps, int H, int W, uint64_t *d_tiles, void *stream);
int trrt_los_batch_tiled(const uint64_t *d_tiles, int n_maps, int H, int W, const int32_t *d_map_id, const int32_t *d_seg,
                         int64_t n, uint8_t *d_out, void *stream);

/* ---------------------------------------------------------------------------
 * K1 nearest_batch.  Replaces the nearest-node scan of rrt.py:156-158
 * (np.argmin over search.L2norm, search.py:13-15): for each integer query
 * point, the index of the tree node with the smallest fp64 squared distance,
 * lowest index on ties.  Tree is SoA: d_x, d_y float64 [n_nodes].
 * d_qxy: int32 [n_q][2].  d_idx: int32 [n_q] (-1 when n_nodes == 0).
 * d_d2: float64 [n_q] squared distance of the winner, or NULL.
 * d_work: scratch of trrt_nearest_workspace_bytes(n_nodes, n_q) bytes.
 * ------------------------------------------------------------------------- */
size_t trrt_nearest_workspace_bytes(int64_t n_nodes, int64_t n_q);
int trrt_nearest_batch(const double *d_x, const double *d_y, int64_t n_nodes, const int32_t *d_qxy, int64_t n_q,
                       int32_t *d_idx, double *d_d2, void *d_work, size_t work_bytes, void *stream);

/* ---------------------------------------------------------------------------
 * K2 rrt_batch.  Replaces rrt.rrt (rrt.py:130-206) and everything it calls:
 * nearest scan (rrt.py:156-158), steer (rrt.py:306-541), drive
 * (rrt.py:272-304), bike_clear / front_of_bike_clear (rrt.py:208-222),
 * search.getArc / getCircle (search.py:96-182), insert / dedupe / goal test
 * (rrt.py:179-201), for n_queries independent (start, goal, sample stream)
 * triples.  rand_conf (rrt.py:53-68) is consumed as an injected stream.
 * K = builtins.K: node capacity, K-1 loop iterations.
 * ------------------------------------------------------------------------- */
typedef struct trrt_rrt_args {
    /* map */
    const uint32_t *d_bits;
    int32_t n_maps, H, W;
    const int32_t *d_map_id; /* [n_queries] or NULL */
    trrt_params params;
    /* queries */
    int64_t n_queries;
    int32_t K;
    int32_t lanes_per_query; /* 0 = auto; else 1,2,4,8,16,32 */
    int32_t schedule;        /* 0 = speculative window of up to `lanes` iterations in one persistent kernel (default),
                                1 = cooperative, one iteration at a time; both give identical results */
    int32_t sample_xy_i16;   /* 0: d_sample_xy is int32 [n_queries][K-1][2]; 1: int16 [n_queries][K-1][2] (coordinates fit: side <= 32768) */
    const double *d_start;   /* [n_queries][3] = x, y, theta_deg (rrt.py:132) */
    const double *d_goal;    /* [n_queries][3]                    (rrt.py:133) */
    const void *d_sample_xy;    /* [n_queries][K-1][2]  rand_conf xy (rrt.py:144), int32 or int16 (sample_xy_i16) */
    const double *d_sample_th;  /* [n_queries][K-1]     rand_conf theta          */
    /* tree outputs, node index = insertion order of G (rrt.py:134-136,180) */
    double *d_node_x;  /* [n_queries][K] */
    double *d_node_y;  /* [n_queries][K] */
    double *d_node_th; /* [n_queries][K] */
    int32_t *d_parent; /* [n_queries][K]  cameFrom[node][0] as index, -1 = none (rrt.py:138,188) */
    double *d_u;       /* [n_queries][K][5] = steer, iccx, iccy, rad, dist of cameFrom[node][1]; NaN icc/rad = straight; may be NULL */
    int32_t *d_n_nodes; /* [n_queries] len(G) (rrt.py:204) */
    int32_t *d_sol;     /* [n_queries] node index of sol or -1 (rrt.py:200) */
    int32_t *d_status;  /* [n_queries] trrt_status */
    int32_t *d_iters;   /* [n_queries] loop iterations executed */
    /* optional per-iteration logs (NULL to skip) */
    int32_t *d_it_near; /* [n_queries][K-1] argmin index (rrt.py:157) or -1 */
    int32_t *d_it_new;  /* [n_queries][K-1] node index of qnew (edge child, rrt.py:185) or -1 */
    uint8_t *d_it_code; /* [n_queries][K-1] trrt_iter_code */
    uint8_t *d_los_log; /* [n_queries][2*(K-1)] search.lineofsight booleans in call order */
    int32_t *d_n_los;   /* [n_queries] */
    uint64_t *d_counters; /* [n_queries][9]: nodes scanned, los calls, los pixels, arc candidate pixels, arc angle tests, steer calls,
                             drive calls, hash probes, nearest decisions where a lower-indexed node has a larger squared distance with the
                             SAME rounded sqrt (the only way argmin(d2) can differ from the reference's argmin(sqrt); expected 0);
                             may be NULL */
    /* scratch */
    void *d_work;
    size_t work_bytes; /* >= trrt_rrt_workspace_bytes(n_queries, K) */
    /* Optional packed copy of the trees (all NULL to skip).  The tree arrays above are [n_queries][K] blocks of which
       only the first n_nodes[q] rows exist (G and cameFrom as rrt.rrt returns them, rrt.py:204-206; about half of K on
       the benchmark workload).  When d_row_start is given, a query that finishes reserves n_nodes[q] consecutive rows of
       the packed arrays with one atomic add on *d_pack_rows and copies its rows there; d_row_start[q] is its first row.
       The caller sets *d_pack_rows to the first row to use before the call (0, or the row where this call's block starts
       inside larger arrays); afterwards it holds the row behind the last one, so the rows of a batch travel to the host
       as ONE linear copy per array.  Queries land in completion order, so row_start is not monotone in q.
       Rows used by a call: sum of n_nodes, at most n_queries * K. */
    uint64_t *d_pack_rows;  /* [1]  next free row */
    int64_t *d_row_start;   /* [n_queries] */
    double *d_pack_x;       /* [rows] */
    double *d_pack_y;
    double *d_pack_th;
    int32_t *d_pack_parent;
    double *d_pack_u;       /* [rows][5]; NULL unless d_u is given too */
} trrt_rrt_args;

size_t trrt_rrt_workspace_bytes(int64_t n_queries, int32_t K);
int trrt_rrt_batch(const trrt_rrt_args *args, void *stream);

/* ---------------------------------------------------------------------------
 * Single-step entry points (batches of independent inputs, one result each);
 * they run the same device functions as the fused kernel.
 *   trrt_steer_batch  replaces rrt.steer (rrt.py:306-541).
 *       d_in  [n][6] = origin x, y, theta, target x, y, theta
 *       d_out [n][8] = landing x, y, theta, steerangle, icc x, icc y, rad, traveldist
 *       d_straight [n] = 1 when the reference returns u = (0, None, None, 1) (rrt.py:541)
 *   trrt_drive_batch  replaces rrt.drive (rrt.py:272-304).
 *       d_in  [n][8] = origin x, y, theta, u.steer, icc x, icc y, rad, dist
 *       d_out [n][3] = final x, y, theta
 *   trrt_arc_batch    replaces `False in [freespace(px) for px in getArc(begin, land, u)]`
 *       (rrt.py:173-174 with search.getArc / getCircle, search.py:96-182).
 *       d_in  [n][9] = begin x, y, land x, y, u.steer, icc x, icc y, rad, straight flag
 *       d_blocked [n] = 1 when some arc pixel is not free.  lanes: 0 = default.
 * ------------------------------------------------------------------------- */
int trrt_steer_batch(const trrt_params *params, int64_t n, const double *d_in, double *d_out, uint8_t *d_straight, void *stream);
int trrt_drive_batch(const trrt_params *params, int64_t n, const double *d_in, double *d_out, void *stream);
int trrt_arc_batch(const uint32_t *d_bits, int n_maps, int H, int W, const int32_t *d_map_id, int64_t n, const double *d_in,
                   uint8_t *d_blocked, int lanes, void *stream);

/* ---------------------------------------------------------------------------
 * Pixel lists of the raster helpers, in the reference's list order, duplicates included:
 *   mode 0  search.getArc(begin, land, u), curved edge    (search.py:144-182)
 *   mode 1  search.bresenham(begin, land), also getArc of a straight u (search.py:43-94, :145-146)
 *   mode 2  search.getCircle(center, r)                   (search.py:96-142; center = icc, r = rad)
 * d_in [n][9] = begin x, y, land x, y, u.steer, icc x, icc y, rad, mode.
 * d_pixels int32 [n][cap][2]; d_count int32 [n] = length of the full list, also when it exceeds cap (call again with a
 * larger cap then).  Only the image shape is needed: getCircle filters by search.valid, not by occupancy.
 *   trrt_clearance_batch  replaces rrt.bike_clear / rrt.front_of_bike_clear (rrt.py:208-222):
 *       d_in [n][3] = x, y, theta -> d_clear uint8 [n][2]
 *   trrt_anglediff_batch  replaces rrt.anglediff (rrt.py:108-115): d_in [n][2] = a1, a2 -> d_out [n]
 * ------------------------------------------------------------------------- */
int trrt_arc_pixels_batch(int H, int W, int64_t n, const double *d_in, int32_t cap, int32_t *d_pixels, int32_t *d_count, void *stream);
int trrt_clearance_batch(const uint32_t *d_bits, int n_maps, int H, int W, const int32_t *d_map_id, const trrt_params *params,
                         int64_t n, const double *d_in, uint8_t *d_clear, void *stream);
int trrt_anglediff_batch(int64_t n, const double *d_in, double *d_out, void *stream);

/* ---------------------------------------------------------------------------
 * rrt.findnearest (rrt.py:117-128): weighted xy+angle nearest over the child
 * entries of G.  Edges are given by the per-iteration log of trrt_rrt_batch
 * (parent = it_near, child = it_new); order of comparison = tree.keys() order
 * then append order, strict `<`.
 * d_best: int32 [n_queries] node index or -1 (reference returns (None, None));
 * d_best_dist: float64 [n_queries].
 * ------------------------------------------------------------------------- */
int trrt_findnearest_batch(const trrt_params *params, int64_t n_queries, int32_t K, const double *d_node_x,
                           const double *d_node_y, const double *d_node_th, const int32_t *d_n_nodes,
                           const int32_t *d_it_near, const int32_t *d_it_new, const double *d_goal, int32_t *d_best,
                           double *d_best_dist, void *stream);

/* ---------------------------------------------------------------------------
 * K3 theta_batch.  Replaces search.astar (search.py:221-307) with
 * getneighbors (search.py:184-194), heuristic / L2norm (search.py:9-15),
 * lazy-Theta* line-of-sight repair (search.py:258-263), reconstruct
 * (search.py:196-204).  thetastar = builtins.THETASTAR (0 gives plain A*).
 * ------------------------------------------------------------------------- */
typedef struct trrt_theta_args {
    const uint32_t *d_bits;
    int32_t n_maps, H, W;
    const int32_t *d_map_id; /* [n_queries] or NULL */
    int32_t thetastar;
    int32_t lanes_per_query; /* 0 = auto; else 8,16,32 */
    int64_t n_queries;
    const int32_t *d_start_goal; /* [n_queries][4] = sx, sy, gx, gy */
    /* outputs */
    int32_t *d_path;     /* [n_queries][path_cap][2] start..goal */
    int32_t path_cap;
    int32_t *d_path_len; /* [n_queries] full length even if > path_cap */
    double *d_cost;      /* [n_queries] sum of L2norm along the path */
    int32_t *d_expanded; /* [n_queries] len(closedSet) when the goal was popped (search.py:270) */
    int32_t *d_status;   /* [n_queries] trrt_status */
    /* optional */
    uint8_t *d_los_log;  /* [n_queries][los_cap] lineofsight booleans in pop order */
    int32_t los_cap;
    int32_t *d_n_los;    /* [n_queries] */
    int32_t *d_pushes;   /* [n_queries] openPQ.put count */
    /* scratch: n_slots concurrent searches, each with H*W cells and heap_cap heap entries */
    int32_t n_slots;     /* 0 = auto */
    int32_t heap_cap;    /* 0 = auto */
    void *d_work;
    size_t work_bytes;
    /* optional dispatch order: slots take query d_order[0], d_order[1], ... (a permutation of 0..n_queries-1).  Searches
       differ in length by orders of magnitude and a batch ends with its longest one, so callers that can guess the
       length (e.g. start-goal distance, longest first) shorten the tail.  Results stay indexed by query.  NULL = 0,1,2,... */
    const int32_t *d_order;
} trrt_theta_args;

/* fills in n_slots / heap_cap when 0 and returns the bytes needed: 256 + n_slots * (H*W + heap_cap) * 16, computed in
   64 bits (default heap_cap = 2*H*W, so 48*H*W bytes per slot: cap n_slots by the memory you can spare before calling);
   0 when the map cannot be planned (2*H*W does not fit an int32: TRRT_ERR_MAP_TOO_LARGE from trrt_theta_batch) */
size_t trrt_theta_workspace_bytes(trrt_theta_args *args);
int trrt_theta_batch(const trrt_theta_args *args, void *stream);

/* ---------------------------------------------------------------------------
 * mission_batch.  Replaces the segment chain of main.py:56-84 (main.chain) for
 * n_missions independent (map, waypoints, sample stream) missions.  Segment s
 * of a mission runs rrt.rrt from waypoint s to s+1 with the headings of
 * main.py:58-67 (rrt.anglebetween, rrt.standardangle); once a segment has
 * failed, every later segment starts at the most recent rrt.findnearest node
 * (rrt.py:117-128) and takes its heading.  Segment s draws its K-1 rand_conf
 * samples (rrt.py:53-68) around its own end from the mission's normals at the
 * current offset, which then advances by 3 * iterations run.
 * A mission stops at segment s, and stop_seg = s, when the RRT status is not
 * OK (TRRT_ERR_REF_RAISES_DRIVE_NONE: the reference raises), when a failed
 * segment has no nearest node (TRRT_ERR_REF_RAISES_NO_NEAREST), or when its
 * normals run out (TRRT_ERR_CAPACITY).  A route whose status is not
 * TRRT_OK_FOUND is copied with zero segments and stop_seg = 0.  A mission that
 * ran its whole chain has status TRRT_OK_FOUND and stop_seg = -1.
 * Each stage s launches a stage kernel, the trrt_rrt_batch launcher over the
 * first n_active[s] slots, and a commit kernel.  Slot i holds mission
 * d_order[i]; callers dispatch missions in decreasing segment count, so that
 * the missions with a segment s are the first n_active[s] slots.
 * ------------------------------------------------------------------------- */
typedef struct trrt_mission_args {
    /* map */
    const uint32_t *d_bits;
    int32_t n_maps, H, W;
    const int32_t *d_map_id;     /* [n_missions] or NULL */
    trrt_params params;
    double xystdv, anglestdv;    /* builtins.xystdv / anglestdv (main.py:31-32), rand_conf rrt.py:53-68 */
    int64_t n_missions;
    int32_t K;                   /* builtins.K: node capacity, K-1 iterations per segment */
    /* routes: the d_path / d_path_len / d_status layout of trrt_theta_batch */
    const int32_t *d_waypoints;  /* [n_missions][wp_cap][2] */
    int32_t wp_cap;
    const int32_t *d_n_waypoints; /* [n_missions]; more than wp_cap -> TRRT_ERR_CAPACITY */
    const int32_t *d_route_status; /* [n_missions] trrt_status of the route search, or NULL (all OK) */
    /* standard normals in draw order: mission m reads d_normals[d_normal_range[m][0] .. d_normal_range[m][1]) */
    const double *d_normals;
    const int64_t *d_normal_range; /* [n_missions][2] */
    /* schedule */
    const int32_t *d_order;      /* [n_missions] slot -> mission */
    int32_t n_stages;
    const int32_t *n_active;     /* HOST [n_stages], non-increasing: missions with a segment s */
    /* per-segment outputs [n_missions][seg_cap]; seg_cap >= the largest segment count (else TRRT_ERR_CAPACITY) */
    int32_t seg_cap;
    double *d_seg_begin;         /* [..][3] x, y, theta of the segment's start */
    double *d_seg_end;           /* [..][3] */
    double *d_seg_solution;      /* [..][3] rrt solution node, NaN when none */
    double *d_seg_nearest;       /* [..][3] findnearest node of a failed segment, NaN otherwise */
    double *d_seg_mindist;       /* [..]    its distance, NaN otherwise */
    int32_t *d_seg_n_nodes;      /* [..] len(G) */
    int32_t *d_seg_n_edges;      /* [..] child entries of G */
    int32_t *d_seg_iters;        /* [..] loop iterations run */
    int32_t *d_seg_status;       /* [..] trrt_status of the segment's RRT, 255 = not run */
    /* per-mission outputs */
    int32_t *d_status;           /* [n_missions] trrt_status */
    int32_t *d_stop_seg;         /* [n_missions] */
    int32_t *d_n_seg;            /* [n_missions] segments of the route */
    double *d_path;              /* [n_missions][path_cap][8] x, y, theta, u[5] of main.path_nodes, segment after segment */
    int32_t *d_path_seg;         /* [n_missions][path_cap] segment of each row */
    int32_t path_cap;
    int32_t *d_path_len;         /* [n_missions] full length even if > path_cap */
    /* scratch, 256-byte aligned */
    void *d_work;
    size_t work_bytes;           /* >= trrt_mission_workspace_bytes(n_missions, K) */
} trrt_mission_args;

/* 19 * 256 + n_missions * (104 + 68 * K + 24 * (K - 1)) + trrt_rrt_workspace_bytes(n_missions, K) */
size_t trrt_mission_workspace_bytes(int64_t n_missions, int32_t K);
int trrt_mission_batch(const trrt_mission_args *args, void *stream);

/* ---------------------------------------------------------------------------
 * legacy_normals.  Seeded sample streams of reference parity: for every seed
 * i, d_out[d_range[i][0] .. d_range[i][1]) receives
 * np.random.RandomState(d_seeds[i]).standard_normal(d_range[i][1] - d_range[i][0])
 * bit for bit (numpy's legacy MT19937 with init_genrand seeding and the polar
 * method of legacy_gauss), the stream rrt.rand_conf (rrt.py:53-68) consumes
 * after np.random.seed(seed).  Ranges must not overlap; empty ones are skipped.
 * numpy takes log(r2) from the host's libm, whose rounding is not correct
 * rounding, so two steps make up one draw:
 *   trrt_legacy_normals_draw   every normal whose libm log is forced by the
 *       error bound of glibc (trrt_libm.h tl_log_decided); an undecided pair
 *       leaves x2 (and x1) in its slots and appends (slot, r2) to the fixup
 *       list: d_fix_pos[k] = slot of f*x2, or ~slot when the pair has no f*x1
 *       slot (odd range); d_fix_r2[k] = r2.  *d_fix_count receives the number
 *       of undecided pairs, also when it exceeds fix_cap (entries past fix_cap
 *       are not written: draw again with a larger list).
 *   trrt_libm_log_batch        HOST: h_out[k] = log(h_in[k]) with this
 *       process's libm, the one numpy's legacy_gauss calls.
 *   trrt_legacy_normals_fixup  the first n_fix <= fix_cap list entries with
 *       d_fix_log[k] = log(d_fix_r2[k]): f = sqrt(-2 log(r2) / r2) and the
 *       pair's slots become f*x2, f*x1.
 * ------------------------------------------------------------------------- */
typedef struct trrt_legacy_normals_args {
    int64_t n_seeds;
    const uint32_t *d_seeds;  /* [n_seeds] */
    const int64_t *d_range;   /* [n_seeds][2] = [begin, end) into d_out */
    double *d_out;
    int64_t *d_fix_pos;       /* [fix_cap] */
    double *d_fix_r2;         /* [fix_cap] */
    int64_t fix_cap;
    uint64_t *d_fix_count;    /* [1] */
    void *d_work;             /* scratch, 256-byte aligned */
    size_t work_bytes;        /* >= trrt_legacy_normals_workspace_bytes(n_seeds) */
} trrt_legacy_normals_args;

size_t trrt_legacy_normals_workspace_bytes(int64_t n_seeds);
int trrt_legacy_normals_draw(const trrt_legacy_normals_args *args, void *stream);
int trrt_libm_log_batch(const double *h_in, double *h_out, int64_t n);
int trrt_legacy_normals_fixup(const trrt_legacy_normals_args *args, const double *d_fix_log, int64_t n_fix, void *stream);

/* ---------------------------------------------------------------------------
 * rand_conf_batch.  rrt.rand_conf (rrt.py:53-68, samples.stream_from_normals)
 * for n queries of n_samples samples each, from standard normals in draw
 * order: query q reads d_normals[q * 3 * n_samples .. (q + 1) * 3 * n_samples)
 * around d_goal[q] = x, y, theta_deg and writes d_sample_xy [n][n_samples][2]
 * (int32, or int16 when sample_xy_i16) and d_sample_th [n][n_samples], the
 * sample layout of trrt_rrt_batch.  Only the map size is needed.
 * ------------------------------------------------------------------------- */
int trrt_rand_conf_batch(int H, int W, double xystdv, double anglestdv, int64_t n, int32_t n_samples, const double *d_goal,
                         const double *d_normals, void *d_sample_xy, int32_t sample_xy_i16, double *d_sample_th, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* THETARRT_H */
