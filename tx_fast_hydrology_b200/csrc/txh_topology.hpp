// txh_topology.hpp -- one-time host pass over the river network.
//
// Replaces the implicit ordering of the reference's headwater walk
// (tx_fast_hydrology/nutils.py:72-88) and `Muskingum.compute_indegree`
// (tx_fast_hydrology/muskingum.py:322-330) by explicit integer artefacts:
// indegree, headwaters, topological levels, level order, unbranched chains,
// the reference's own visit sequence (test hook), and the dataflow schedule
// the persistent routing kernel consumes.  Pure C++17, no CUDA, exact integers.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

namespace txh {

struct Topology {
    int64_t n = 0;
    std::vector<int32_t> end;         // downstream reach; self-loop at outlets
    std::vector<int32_t> indeg;       // muskingum.py:322-330 (self-loops excluded)
    std::vector<int32_t> child_off;   // CSR of upstream reaches, ascending id
    std::vector<int32_t> child;
    std::vector<int32_t> heads;       // indegree == 0, ascending (muskingum.py:444)
    std::vector<int32_t> topo;        // a topological order (Kahn, by level then id)
    std::vector<int32_t> level;       // 0 at headwaters, else 1 + max(level[upstream])
    int32_t nlevels = 0;
    std::vector<int32_t> level_off;   // reaches of level l are topo[level_off[l]..level_off[l+1])
    std::vector<int32_t> subtree;     // reaches draining through j (inclusive)
    std::vector<int32_t> main_child;  // upstream reach of highest level (ties: lowest id), -1 at headwaters
    std::vector<int32_t> path_id;     // longest-path decomposition: path index of each reach
    std::vector<int32_t> path_pos;    // position along the path, 0 at the headwater
    std::vector<int32_t> path_len;    // per path
    std::vector<int32_t> chain_id;    // maximal unbranched runs (u -> v with indegree[v] == 1)
    std::vector<int32_t> chain_pos;
    std::vector<int32_t> chain_len;   // per chain
    std::vector<int32_t> visit;       // order in which nutils.py:72-88 evaluates reaches

    bool build(int64_t n_, const int64_t* endnodes, std::string& err);
};

struct SchedParams {
    int long_path_min = 64;   // paths at least this long become spines
    int spine_cap = 0;        // reaches per spine segment; 0 = chosen from the depth of the network (6..16)
    int pocket_cap = 16;      // reaches per pocket task (bundled side subtrees)
    int max_slots = 8;        // shared-memory scratch rows per warp
    int link_cap = 8;         // segments per LINK task (dataflow kernel: blocks chained along the path)
    int side_cap = 10;        // pocket roots joining one spine segment (its serial work per step paces the chain)
};

// Per-reach header word consumed by the routing kernel.
//   pocket rows : bit 0      inflow starts from the running accumulator (previous reach's outflow)
//                 bits 1..5  (scratch slot + 1) the outflow is also parked in, 0 = none
//                 bits 6..30 number of input words that follow in the task's input stream
//                 bit 31     pocket root feeding a spine: one more word follows, the row of the
//                            side buffer the outflow is also pushed to (read back by that
//                            segment's PRE as a contiguous slab instead of a gather)
//   spine rows  : bit 0      not the first reach of its segment (the recurrence continues)
//                 bits 6..18 number of side-buffer rows the reach consumes (its pocket roots, in
//                            the order the PRE task walks them, starting at TaskDesc::side_off)
//                 bits 19..31 first row of a segment only: number of rows whose sum is the flow
//                             entering the segment (last row of the upstream segment + outlets of
//                             long tributaries; FIX task stream)
// Input word: bit 31 set -> state row (position) to gather; else scratch slot id.
// LINK stream, one record per segment of the path: [last row position][n_late][n_late rows].
constexpr uint32_t HDR_ACC = 1u;
constexpr uint32_t HDR_PUSH = 0x80000000u;
constexpr uint32_t INW_ROW = 0x80000000u;
constexpr int TASK_POCKET = 0, TASK_PRE = 1, TASK_LINK = 2, TASK_FIX = 3;

// Dataflow task.  A task T may run step s once (a) every task in A(T) has finished step s and
// (b) every task in B(T) (T itself included) has finished step s-1.  Completion of U at step s
// decrements the pending counter of every T with U in A(T) ("same" targets, for T's step s) and
// of every T with U in B(T) ("next" targets, for T's step s+1).
//
// Spines (long paths) are cut into segments.  Along a segment the step is the recurrence
// o_k = alpha_k (o_{k-1} + side_k) + r_k, an affine map of the flow o_in entering the segment:
//   PRE   per segment : side_k, r_k from the old state and the pocket roots; B_k = the recurrence
//                       with o_in = 0; parks (side_k, B_k) in the segment's I / O rows
//   LINK  per block of consecutive segments, chained along the path: out = A_last * o_in + B_last
//                       (A = prefix product of alpha), one FMA per segment on the critical path
//   FIX   per segment : o_k = B_k + A_k * o_in, i_k = o_{k-1} + side_k, all reaches independent
struct TaskDesc {
    int32_t begin;     // first position (rows [begin, begin+len) are contiguous); LINK: first link entry
    int32_t len;       // rows; LINK: segments of the path
    int32_t in_off;    // offset of the task's first input word
    int32_t nfy_off;   // offset into `notify`: n_same targets, then n_next targets
    int32_t n_same;
    int32_t n_next;
    int32_t need0;     // |A(T)|           pending count before step 0
    int32_t need;      // |A(T)| + |B(T)|  re-arm value after each completed step
    int32_t kind;      // TASK_POCKET / TASK_PRE / TASK_LINK / TASK_FIX
    int32_t n_words;   // input words of this task
    int32_t side_off;  // PRE: first side-buffer row of the segment
    int32_t pad_;
};

// Window task (route_window_kernel): one warp owns the task's rows in shared memory for every step of
// a launch and exchanges single rows with other tasks through the slot ring.
//   WPOCKET : a pocket (bundled side subtrees), evaluated depth-first each step
//   WSEG    : one spine segment; per step the PRE recurrence, the hop
//             out = A_last * o_in + B_last published to its own slot, then the FIX pass
// Input word (window mode): bit 31 -> slot of the ring, bit 30 -> row of this task, else scratch slot.
// Stream of a WPOCKET: the words of its rows in order (a row whose header has HDR_PUSH is followed by
// the slot it publishes).  Stream of a WSEG: [n_in entering slots][side slots of the rows in order].
constexpr uint32_t WIN_SLOT = 0x80000000u, WIN_OWN = 0x40000000u;
constexpr int WTASK_POCKET = 0, WTASK_SEG = 1;
struct WTaskDesc {
    int32_t begin, len;      // rows [begin, begin + len)
    int32_t kind;
    int32_t in_off, n_words; // input stream
    int32_t prod_off, n_prod;// producer tasks (indices in window-task order, all smaller than this task's): first the
                             // n_in owners of the entering slots (same order), then the distinct other producers
    int32_t out_slot;        // WSEG: slot of the segment's outflow; -1 otherwise
    int32_t n_in;            // WSEG: number of entering slots at the head of the stream
    int32_t n_out;           // rows this task publishes per step (0: nobody waits for it)
    int32_t n_own;           // input words that read a row of the task itself (scratch-slot fallback)
    int32_t pad_;
};

// ---------------------------------------------------------------------------------------------------
// Lane schedule (route_lane_kernel, small ensembles): lanes are REACHES, not members.
//
// The network is cut into regions (unions of sub-trees); one CTA owns a region for every step of a launch
// with its state in shared memory.  Inside a region every row (reach) has a skew offset
//   off = D - d,   d = distance (in reaches) to the exit of its sub-tree, D = the sub-tree's largest d,
// and evaluates timestep s in iteration k = s + off of the CTA's loop.  An edge u -> j inside a region then
// has off[u] = off[j] - 1: what a row reads in iteration k was written in iteration k - 1, one barrier apart,
// so ALL rows of a region are busy in every iteration, each on its own timestep (time skewing, SURVEY.md
// appendix B).  Outflows that cross regions travel through per-(slot, member) streams in global memory,
// ring[slot][member][step]; the consuming region mirrors every stream as a VIRTUAL row (a leaf one skew level
// above its consumer) whose thread copies the stream into the row buffer, prefetching 16 steps ahead.
// Regions are claimed in a topological order of the region graph (producers first).
struct LaneRegionDesc {
    int32_t row_off;      // first entry of this region in the row arrays (real rows, then virtual rows)
    int32_t n_real;
    int32_t n_virt;
    int32_t child_off;    // first entry in `child` (children beyond the two a row record carries inline)
    int32_t n_child;
    int32_t n_extra;      // largest skew offset + 1: iterations of a launch = nsteps + n_extra - 1
    int32_t height;       // level of the region in the region graph (0: depends on no other region)
    int32_t pad_;
};
constexpr int kLaneMaxRows = 896;    // rows of a region: one per thread of a 1,024-thread CTA, the rest mirror streams

struct LaneSchedule {
    int mt = 0;                             // member tile the regions were sized for (1, 2, 4, 8, 16)
    int cap_rows = 0;
    size_t smem_budget = 0;
    std::vector<LaneRegionDesc> regions;    // ticket order
    // per row (region-local order): reach id (-1: virtual), skew offset, the first two children c0 | c1 << 16
    // (region-local rows; a missing child is the region's ZERO row, index n_real + n_virt), the number of further
    // children and where they start in `child` (relative to the region's child_off), slot (real: stream the
    // outflow is published to, or -1; virtual: stream it mirrors).
    // Rows are ordered by (has further children, skew offset, position): the lanes of a warp then sit on (nearly)
    // the same timestep, so their per-step records are one broadcast load and they change forcing bracket together.
    std::vector<int32_t> row_reach, row_off, row_c01, row_nx, row_xbeg, row_slot;
    std::vector<uint16_t> child;            // region-local row indices (children beyond the first two)
    int32_t n_slots = 0, max_real = 0, max_virt = 0, max_child = 0, max_extra = 0;
    size_t max_bytes = 0;                   // shared memory of the largest region

    // bytes of shared memory a region of (real, virt, child) rows needs at member tile mt
    static size_t region_bytes(size_t real, size_t virt, size_t nchild, int mt);
    // side_min: side tributaries of at least this many rows always become clusters of their own
    bool build(const Topology& t, const std::vector<int32_t>& pos_of_reach, int mt, int cap_rows, size_t smem_budget,
               int side_min, std::string& err);
};

struct Schedule {
    SchedParams prm;
    std::vector<int32_t> pos_of_reach, reach_of_pos;
    std::vector<TaskDesc> tasks;            // in a topological (critical-path-first) order of the A-edges
    std::vector<int32_t> notify;
    std::vector<int32_t> init_ready;        // tasks with need0 == 0
    std::vector<uint32_t> hdr;              // per position
    std::vector<uint32_t> inw;
    std::vector<int32_t> link_last;         // per LINK entry: position of the segment's last row
    // position-space CSR of upstream rows (level kernel, init_inflows, apply_gain)
    std::vector<int32_t> up_off, up_pos;
    std::vector<int32_t> lvl_pos, lvl_off;  // positions sorted by level
    std::vector<uint8_t> is_outlet_pos;
    // statistics
    int32_t n_spine = 0, n_pocket = 0, slots_used = 0, row_fallbacks = 0;
    int32_t max_len = 0;                    // longest POCKET / PRE / FIX task (rows)
    int32_t max_link_len = 0;               // longest LINK task (segments)
    int32_t max_words = 0, max_link_words = 0;   // longest input streams (walking tasks / LINK)
    int32_t n_side = 0;                     // rows of the side buffer
    // window-mode descriptors over the same row layout
    std::vector<WTaskDesc> wtasks;          // in a topological, critical-path-first order
    std::vector<uint32_t> whdr, winw;       // per-position headers / input streams of the window tasks
    std::vector<int32_t> wprod;
    int32_t n_wslots = 0, w_max_len = 0, w_max_words = 0, w_max_prod = 0, w_cp_tasks = 0, w_n_own = 0;
    int32_t cp_tasks = 0;                   // tasks on the longest same-step dependent chain
    int64_t cp_cost = 0;

    bool build(const Topology& t, const SchedParams& p, std::string& err);
};

}  // namespace txh
