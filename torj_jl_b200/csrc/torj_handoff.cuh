// Segment hand-off protocol of k_trace: the per-ray word seg_done[ray] and its two transitions.
//
// Under the hand-off schedule work item i is segment i / n of ray i % n (shifted by the ray's predicted life with
// life-ordered rounds), and items are drawn in queue order but may be CLAIMED in any order: a warp that drew an item early
// can reach its claim after a warp that drew a later item. Nobody waits for an unfinished predecessor. A claim whose
// segment cannot start yet is dropped and marked in the word; the lane running the ray finds the mark when it hands its
// segment in and continues with the ray itself. Every change to the word goes through one of the two pure functions below,
// applied with compare-and-swap, so that for every order of claims and hand-ins each segment of a ray runs exactly once
// and nothing is left that can never run (tests/test_handoff_protocol.py checks this for every interleaving).
//
// Word layout (a live word is never TORJ_SEG_RETIRED: DONE <= TORJ_SEG_MAX < 0x7fff):
//   bits  0-14  DONE: segments completed (handed in)
//   bits 15-29  DROP: 1 + the highest segment whose item was dropped because it was claimed before it could start
//   bit  30     RUNNING: a lane holds segment DONE (claimed it, or continues with it after a hand-in)
//   TORJ_SEG_RETIRED once the ray has ended.
// Plain C++ with no CUDA dependency beyond the __host__ __device__ qualifier, so the host can test the same code.
#pragma once

#ifdef __CUDACC__
#define TORJ_HD __host__ __device__ __forceinline__
#else
#define TORJ_HD inline
#endif

#define TORJ_SEG_RETIRED 0x7fffffff
#define TORJ_SEG_RUNNING (1 << 30)
#define TORJ_SEG_MAX 16000  // n_segments the 15-bit fields are used for under the hand-off
#define TORJ_SEG_DONE(w) ((w) & 0x7fff)
#define TORJ_SEG_DROP(w) (((w) >> 15) & 0x7fff)

struct TorjSegMove {
    int w;   // the word after the transition (equal to the input: nothing to write)
    int go;  // claim: the item is ready, the claiming lane runs segment wseg; hand-in: the lane continues with the ray
};

// A lane claims the item of segment wseg (0-based) of a ray whose word is w.
TORJ_HD TorjSegMove torj_seg_claim(int w, int wseg) {
    if (w == TORJ_SEG_RETIRED || TORJ_SEG_DONE(w) > wseg) return {w, 0};  // the ray has ended / the segment has run
    if (TORJ_SEG_DONE(w) == wseg) {
        if (w & TORJ_SEG_RUNNING) return {w, 0};  // the previous holder continues with this segment
        return {w | TORJ_SEG_RUNNING, 1};
    }
    // the ray's previous segment is still running: drop the item and leave the segment to its holder
    const int drop = TORJ_SEG_DROP(w) > wseg + 1 ? TORJ_SEG_DROP(w) : wseg + 1;
    return {(w & (TORJ_SEG_RUNNING | 0x7fff)) | (drop << 15), 0};
}

// The holder of a ray hands in its segment seg - 1 (seg = segments begun, 1-based) without retiring the ray. It continues
// with segment seg itself when that segment's item was dropped; otherwise the item's claim will start it.
TORJ_HD TorjSegMove torj_seg_hand_in(int w, int seg) {
    const int go = TORJ_SEG_DROP(w) >= seg + 1;
    return {((w & ~TORJ_SEG_RUNNING) + 1) | (go ? TORJ_SEG_RUNNING : 0), go};
}
