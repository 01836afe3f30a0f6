/* spn_tracks.h - multi-view feature tracks from verified matches (part of libspn_b200.so).
 *
 * A track is the set of keypoints, one per image, that see the same 3-D point.  spn_track_labels takes the connected
 * components of the graph whose nodes are the keypoints of a collection and whose edges are its kept matches (GLOMAP /
 * OpenMVG build tracks this way); spn_track_table turns the component labels into a track table.
 *
 * Conventions are those of spn_b200.h: return 0 or a negative SPN_E_* code with spn_last_error(), caller-owned device
 * buffers, work enqueued on `stream`.  Scratch lives in the context's guard-banded scratch buffer (spn_check_guards).
 *
 * The rule (oracle/tracks_oracle.py restates it with scipy):
 *   - Nodes are the rows r of the keypoint table of features.npz: image n's keypoint i is r = offsets[n] + i, so there
 *     are K = offsets[N] nodes, 1 <= K <= 2^31 - 1.
 *   - Edges.  A kept match (i, j) of the pair (a, b) is the edge (offsets[a] + i, offsets[b] + j).  Duplicate edges and
 *     self-loops are allowed and change nothing.
 *   - Label.  A node's label is the smallest row of its connected component.  It does not depend on the order of the
 *     edges, on thread scheduling or on how the edges are split over calls: the outputs are bit-identical whenever the
 *     set of edges is.
 *   - Tracks are the components of at least min_length nodes, ordered by label; a track's observations are its rows in
 *     ascending order, which is image order.  A track is consistent iff no two of its observations lie in one image.
 *     Inconsistent tracks are flagged, not split or dropped.
 *
 * spn_track_labels(ctx, d_edges, E, K, resume, d_label, d_bad, stream)
 *   d_edges [E][2]   int32 (row, row); may be NULL when E == 0
 *   resume           0: the labels start as singletons (label[r] = r); 1: d_label holds the labels of an earlier call
 *                    with the same K and the edges are joined into those components, so splitting an edge list over
 *                    several calls gives the labels of one call over all of it
 *   d_label [K]      int32 out: the label of every row
 *   d_bad [1]        int64 out: the edges with an endpoint outside [0, K), which are not applied, plus (resume only) the
 *                    input labels outside [0, r], which are reset to r first
 *   Algorithm: union-find after ECL-CC (Jaiganesh & Burtscher 2018).  A root only ever hooks under a smaller root with
 *   atomicCAS, finds halve their path, and a last pass writes label[r] = find(r); since roots only point to smaller
 *   rows, the root of a component is its minimum.  E is 64-bit: there is no per-call limit on the edges.
 *
 * spn_track_table(ctx, d_label, K, d_img_offsets, N, min_length, d_track_offsets, d_obs, d_consistent, d_track_of,
 *                 d_totals, d_bad, stream)
 *   d_label [K]              int32: spn_track_labels' output
 *   d_img_offsets [N+1]      int64: image n's rows are offsets[n] .. offsets[n+1] - 1 (offsets[0] = 0, non-decreasing,
 *                            offsets[N] = K);  1 <= N <= 2^31 - 2
 *   min_length               >= 2 nodes per track (so a singleton is never a track)
 * Outputs, allocated at their upper bounds T <= K / 2 and O <= K (only the first T (+1) / O entries are written):
 *   d_track_offsets [K/2+1]  int64: track t's observations are d_obs[offsets[t] .. offsets[t+1] - 1]
 *   d_obs [K][2]             int32 (image, keypoint) of every observation, tracks in label order, rows ascending
 *   d_consistent [K/2]       uint8 1 iff the track has no two observations in one image
 *   d_track_of [K]           int32 track of every row, -1 for rows in no track
 *   d_totals [2]             int64 (T, O): the number of tracks and of observations
 *   d_bad [1]                int64: rows whose label is not a label of spn_track_labels (outside [0, r], or pointing
 *                            at a row that is not its own label; such rows are in no track) plus image offsets that
 *                            break the conditions above (counted, not repaired: the observations are then undefined)
 *   The observation order comes from a stable radix sort of the rows by track (CUB's DeviceRadixSort, header-only), so
 *   no atomic decides it; component sizes use integer atomics, whose totals do not depend on their order.
 *   Scratch: 24 K bytes plus the sort's temporary storage.
 */
#ifndef SPN_TRACKS_H
#define SPN_TRACKS_H

#include "spn_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

SPN_API int spn_track_labels(spn_ctx* ctx, const int32_t* d_edges, int64_t E, int32_t K, int resume, int32_t* d_label,
                             int64_t* d_bad, spn_stream stream);

SPN_API int spn_track_table(spn_ctx* ctx, const int32_t* d_label, int32_t K, const int64_t* d_img_offsets, int32_t N,
                            int32_t min_length, int64_t* d_track_offsets, int32_t* d_obs, uint8_t* d_consistent,
                            int32_t* d_track_of, int64_t* d_totals, int64_t* d_bad, spn_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SPN_TRACKS_H */
