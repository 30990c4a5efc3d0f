// Stage 2b: person proposals from edge-node scores, one warp per frame.
//
// Reference behaviour restated (utils/skeleton_matching_utils.py):
//   :32-55   walk the edges in id order: heads enter the proposal graph when first seen as the
//            destination of an edge leaving an edge-node; an edge-node whose score is > threshold
//            (strict) becomes a Matching(nodes=list({h1,h2}))  -> order of the pair = CPython set order
//   :60      stable sort by score, descending (ties keep edge-node order)
//   :61-108  greedy camera-exclusive merge with per-head linked-camera lists and per-group camera
//            lists; merging two groups relabels the absorbed one and FORGETS its cameras (:97-102)
//   :117-130 nx.connected_components (BFS in node-insertion order), components smaller than
//            min_number_of_views dropped, person[camera] = head for every head in the component's
//            *set iteration order* (matters when a component holds two heads of one camera)
//
// Camera lists are only ever tested for membership, so they are 32-bit camera masks. The CPython
// set layout (Objects/setobject.c: table of 8, LINEAR_PROBES 9, PERTURB_SHIFT 5, growth when
// fill*5 >= mask*3 to the first power of two > 4*used) is emulated exactly; connected components
// are labelled by a level-order BFS over the link list in insertion order, which is what
// networkx 3.x _plain_bfs does.
#include "common.cuh"

namespace b200pose {

__device__ __forceinline__ uint32_t ordered_bits(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// CPython set insert of small non-negative ints (hash(i) == i). Returns true if inserted.
__device__ bool set_probe_insert(int* table, int mask, int key) {
    unsigned perturb = (unsigned)key;
    int i = key & mask;
    while (true) {
        if (table[i] < 0) { table[i] = key; return true; }
        if (table[i] == key) return false;
        if (i + 9 <= mask) {
            for (int j = 1; j <= 9; ++j) {
                if (table[i + j] < 0) { table[i + j] = key; return true; }
                if (table[i + j] == key) return false;
            }
        }
        perturb >>= 5;
        i = (int)(((unsigned)i * 5u + 1u + perturb) & (unsigned)mask);
    }
}

struct IntSet {
    int* tab;      // current table
    int* spare;    // scratch for growth
    int mask;
    int fill;
    __device__ void init(int* a, int* b) {
        tab = a; spare = b; mask = 7; fill = 0;
        for (int i = 0; i < 8; ++i) tab[i] = -1;
    }
    __device__ void add(int key) {
        if (!set_probe_insert(tab, mask, key)) return;
        ++fill;
        if (fill * 5 < mask * 3) return;
        const int minused = fill * 4;
        int newsize = 8;
        while (newsize <= minused) newsize <<= 1;
        for (int i = 0; i < newsize; ++i) spare[i] = -1;
        for (int i = 0; i <= mask; ++i)
            if (tab[i] >= 0) set_probe_insert(spare, newsize - 1, tab[i]);
        int* t = tab; tab = spare; spare = t;
        mask = newsize - 1;
    }
};

__device__ __forceinline__ void pair_order(int h1, int h2, int& a, int& b) {
    // list({h1, h2}) for a set built as set([h1]); add(h2): slot order in a table of 8
    const int s1 = h1 & 7;
    int i = h2 & 7;
    unsigned perturb = (unsigned)h2;
    while (i == s1) {
        perturb >>= 5;
        i = (int)(((unsigned)i * 5u + 1u + perturb) & 7u);
    }
    if (s1 < i) { a = h1; b = h2; } else { a = h2; b = h1; }
}

struct ClusterParams {
    const int* head_off; const int* node_off; const int* pairs; const int* node_cam; const float* scores;
    int v_sm; double threshold; int min_views;
    int* person_heads; int* n_persons;
    int max_heads, max_keys, table_cap;
    int general;    // 1: edge-node list without closed form (b200pose_build_graph_pairs): first-seen order from the pairs
};

// blockDim = 32 (frames of a few hundred edge-nodes: everything is warp-synchronous) or 256 / 1024 (large frames: the sort
// and the table passes use the whole CTA; the order-dependent parts still run on one lane).
// The second launch bound sets the register budget: 64 for the 256-thread instantiation (4 CTAs), whose rank sort keeps 16
// keys and 16 ranks per lane in registers (ptxas's own choice, 40, spills them), and 32 for the 1024-thread one (2 CTAs).
template <int MAXT>
__global__ void __launch_bounds__(MAXT, MAXT == 256 ? 4 : 2) cluster_kernel(ClusterParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int n_seen_s, n_valid_s, n_links_s;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int lane = tid & 31;
    const bool one_warp = nt == 32;
    auto bsync = [&]() { if (one_warp) __syncwarp(); else __syncthreads(); };
    const int b = blockIdx.x;
    const int h0 = p.head_off[b];
    const int H = p.head_off[b + 1] - h0;
    const int n0 = p.node_off[b];
    const int M = p.node_off[b + 1] - n0 - H;
    const int m0 = n0 - h0;
    // ---- carve shared memory ----
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);
    int* link_a = reinterpret_cast<int*>(keys);                     // links alias the consumed front of keys
    int* ip = reinterpret_cast<int*>(keys + p.max_keys);
    int* cam = ip;              ip += p.max_heads;
    int* group = ip;            ip += p.max_heads;
    int* first_seen = ip;       ip += p.max_heads;
    int* queue = ip;            ip += p.max_heads;
    unsigned* linked = reinterpret_cast<unsigned*>(ip); ip += p.max_heads;
    unsigned* cams_for = reinterpret_cast<unsigned*>(ip); ip += p.max_heads;
    int* flag = ip;             ip += p.max_heads;
    int* tab_a = ip;            ip += p.table_cap;
    int* tab_b = ip;

    if (H > p.max_heads || M > p.max_keys || H == 0) {              // outside the sized limits: no persons
        if (tid == 0) p.n_persons[b] = 0;
        return;
    }
    int Mpad = 1;
    while (Mpad < M) Mpad <<= 1;

    for (int h = tid; h < H; h += nt) {
        cam[h] = p.node_cam[n0 + h];
        group[h] = -1;
        linked[h] = 1u << cam[h];
        flag[h] = 0;
    }
    // ---- matchings above the threshold (:49-55): sort key = (score, edge-node index descending) ----
    // Small frames (one warp, <= 512 edge-nodes): the keys above the threshold are compacted with a ballot prefix and
    // rank-sorted - every lane counts, for each of its keys, how many keys are greater (broadcast reads, no dependent
    // chain) - instead of 36 dependent passes of a padded bitonic network, which took half of this kernel.
    const bool rank_sort = MAXT <= 256 && one_warp && p.max_keys <= 512;
    int n_valid = 0;
    if (rank_sort) {
        for (int k0 = 0; k0 < M; k0 += 32) {
            const int k = k0 + lane;
            unsigned long long key = 0ull;
            if (k < M) {
                const float s = p.scores[n0 + H + k];
                if ((double)s > p.threshold)
                    key = ((unsigned long long)ordered_bits(s) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)k);
            }
            const unsigned bal = __ballot_sync(0xffffffffu, key != 0ull);
            if (key != 0ull) keys[n_valid + __popc(bal & ((1u << lane) - 1u))] = key;
            n_valid += __popc(bal);
        }
        __syncwarp();
    } else {
        // Large frames: only the matchings above the threshold are kept (a 10-view x 16-person frame has 11520
        // edge-nodes and ~720 matchings), in any order - the keys are unique and the sort below orders them - so the
        // bitonic network runs over the next power of two of the survivors instead of over every edge-node.
        if (tid == 0) n_valid_s = 0;
        __syncthreads();
        for (int k = tid; k < M; k += nt) {
            const float s = p.scores[n0 + H + k];
            if ((double)s > p.threshold)
                keys[atomicAdd(&n_valid_s, 1)] = ((unsigned long long)ordered_bits(s) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)k);
        }
        __syncthreads();
        n_valid = n_valid_s;
        Mpad = 2;
        while (Mpad < n_valid) Mpad <<= 1;
        if (Mpad > p.max_keys) Mpad = p.max_keys;
        for (int k = n_valid + tid; k < Mpad; k += nt) keys[k] = 0ull;
    }
    bsync();
    // ---- first-seen order of the heads in the reference's edge walk (:32-47), in closed form. Edge-nodes are ordered
    // by camera-group pair (g0,g1), (g0,g2), ..., (g1,g2), ... and, inside a pair, head1-major; an edge-node shows its
    // head1 before its head2. With a = heads of g0 and b = heads of g1 the walk therefore meets a0, b0, b1, ..., then
    // a1, a2, ..., then the heads of g2, g3, ... in index order; heads are numbered group by group, so
    //     first_seen = [0, n0 .. n0+n1-1, 1 .. n0-1, n0+n1 .. H-1]          (n0, n1 = sizes of the first two groups)
    // and a frame whose heads all sit in one camera has no edge-node and sees nothing. ----
    if (p.general) {
        // explicit edge-node list: the walk (:32-47) meets, per edge-node in order, its head1 then its head2, so a head's
        // first appearance is its smallest position in the flattened pair list, and the first-seen order is the heads
        // sorted by that position (rank by counting: positions are distinct)
        for (int h = tid; h < H; h += nt) flag[h] = 0x7fffffff;
        bsync();
        for (int t = tid; t < 2 * M; t += nt) {
            const unsigned h = (unsigned)p.pairs[2 * (size_t)m0 + t];
            if (h < (unsigned)H) atomicMin(&flag[h], t);
        }
        bsync();
        if (tid == 0) n_seen_s = 0;
        bsync();
        for (int h = tid; h < H; h += nt) {
            const int mine = flag[h];
            if (mine == 0x7fffffff) continue;
            int r = 0;
            for (int o = 0; o < H; ++o) r += flag[o] < mine ? 1 : 0;
            first_seen[r] = h;
            atomicAdd(&n_seen_s, 1);
        }
        bsync();
        for (int h = tid; h < H; h += nt) flag[h] = 0;
    } else if (tid == 0) {
        int n0g = 1;
        while (n0g < H && cam[n0g] == cam[0]) ++n0g;
        int n_seen = 0;
        if (n0g < H && M > 0) {
            int n1g = 1;
            while (n0g + n1g < H && cam[n0g + n1g] == cam[n0g]) ++n1g;
            first_seen[n_seen++] = 0;
            for (int i = 0; i < n1g; ++i) first_seen[n_seen++] = n0g + i;
            for (int i = 1; i < n0g; ++i) first_seen[n_seen++] = i;
            for (int i = n0g + n1g; i < H; ++i) first_seen[n_seen++] = i;
        }
        n_seen_s = n_seen;
    }
    bsync();
    const int n_seen = n_seen_s;

    if constexpr (MAXT <= 256) if (rank_sort) {
        // ---- rank sort, descending (keys are unique: the edge-node index is part of the key) ----
        unsigned long long mine[16];
        int rank[16];
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const int idx = lane + 32 * r;
            mine[r] = idx < n_valid ? keys[idx] : 0ull;
            rank[r] = 0;
        }
        const int R = (n_valid + 31) >> 5;                           // key slots in use per lane (uniform)
        for (int j = 0; j < n_valid; ++j) {
            const unsigned long long kj = keys[j];
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                if (r >= R) break;
                rank[r] += (kj > mine[r]) ? 1 : 0;
            }
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 16; ++r)
            if (lane + 32 * r < n_valid) keys[rank[r]] = mine[r];
        if (lane == 0 && n_valid < p.max_keys) keys[n_valid] = 0ull;     // terminates the merge walk
        __syncwarp();
    }
    if (!rank_sort) {
    // ---- bitonic sort, descending: score desc, edge-node index asc (:60) ----
    for (int size = 2; size <= Mpad; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = tid; i < Mpad; i += nt) {
                const int j = i ^ stride;
                if (j > i) {
                    const unsigned long long x = keys[i], y = keys[j];
                    const bool desc = ((i & size) == 0);
                    if (desc ? (x < y) : (x > y)) { keys[i] = y; keys[j] = x; }
                }
            }
            bsync();
        }
    }
    }
    // ---- replace every sorted key by its (h1, h2) pair: one parallel pass of coalesced-ish global reads, so the
    // sequential merge below touches shared memory only ----
    for (int t = tid; t < (rank_sort ? n_valid : Mpad); t += nt) {
        const unsigned long long key = keys[t];
        if (key != 0ull) {
            const int k = (int)(0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull));
            const unsigned long long h1 = (unsigned long long)p.pairs[2 * (m0 + k)], h2 = (unsigned long long)p.pairs[2 * (m0 + k) + 1];
            keys[t] = (1ull << 63) | (h1 << 31) | h2;
        }
    }
    bsync();

    // ---- greedy merge (:61-108): inherently sequential in score order. Warp 0 takes the sorted matchings 32 at a
    // time: every lane runs the three rejection tests (:67, :70-75) on its matching against the state as it stands,
    // and lane 0 then walks the survivors in order with the full set of tests. A rejected matching changes nothing,
    // and between two group absorptions the state only grows (linked-camera masks and group camera masks gain bits, a
    // head's group never changes once set), so a matching rejected now is rejected at its turn too. An absorption
    // (:90-104) forgets the absorbed group's cameras, which can revive a matching: the rest of the batch is then
    // tested again. A 10-view x 16-person frame has ~8000 matchings above the threshold and ~140 links; the walk used
    // to be one lane over all of them. ----
    int n_links = 0;
    if (tid < 32) {
        int cur = 0;
        bool done = false;
        for (int t0 = 0; t0 < n_valid && !done; t0 += 32) {
            const int t = t0 + lane;
            const unsigned long long key = t < n_valid ? keys[t] : 0ull;
            int a = 0, c = 0;
            unsigned ca = 0, cc = 0;
            if (key != 0ull) {
                const int h1 = (int)((key >> 31) & 0x7FFFFFFFull), h2 = (int)(key & 0x7FFFFFFFull);
                pair_order(h1, h2, a, c);
                ca = 1u << cam[a]; cc = 1u << cam[c];
            }
            done = __any_sync(0xffffffffu, t < n_valid && key == 0ull);       // the zero key ends the walk
            unsigned pending = __ballot_sync(0xffffffffu, key != 0ull);
            while (pending) {
                bool alive = false;
                if ((pending >> lane) & 1u) {
                    alive = !((ca & linked[c]) || (cc & linked[a]));                            // :67
                    if (alive) {
                        const int ga = group[a], gc = group[c];
                        if (ga >= 0 && (cc & cams_for[ga])) alive = false;                      // :70-72
                        else if (gc >= 0 && (ca & cams_for[gc])) alive = false;                 // :73-75
                        else if (ga >= 0 && gc >= 0 && (cams_for[gc] & cams_for[ga])) alive = false;   // :91
                    }
                }
                unsigned bal = __ballot_sync(0xffffffffu, alive);
                pending = 0u;
                while (bal) {
                    const int src = __ffs(bal) - 1;
                    bal &= bal - 1;
                    const int xa = __shfl_sync(0xffffffffu, a, src), xc = __shfl_sync(0xffffffffu, c, src);
                    const unsigned xca = __shfl_sync(0xffffffffu, ca, src), xcc = __shfl_sync(0xffffffffu, cc, src);
                    int absorbed = 0;
                    if (lane == 0) {
                        do {
                            if ((xca & linked[xc]) || (xcc & linked[xa])) break;                  // :67
                            const int ga = group[xa], gc = group[xc];
                            if (ga >= 0 && (xcc & cams_for[ga])) break;                         // :70-72
                            if (gc >= 0 && (xca & cams_for[gc])) break;                         // :73-75
                            if (ga < 0 && gc < 0) {                                             // :77-83
                                group[xa] = cur; group[xc] = cur; cams_for[cur] = xca | xcc;
                                ++cur;
                            } else if (ga >= 0 && gc < 0) {                                     // :84-86
                                group[xc] = ga; cams_for[ga] |= xcc;
                            } else if (gc >= 0 && ga < 0) {                                     // :87-89
                                group[xa] = gc; cams_for[gc] |= xca;
                            } else {                                                            // :90-104
                                if (cams_for[gc] & cams_for[ga]) break;
                                for (int h = 0; h < H; ++h)
                                    if (group[h] == gc) group[h] = ga;                          // absorbed cameras are forgotten
                                absorbed = 1;
                            }
                            link_a[2 * n_links] = xa; link_a[2 * n_links + 1] = xc;             // :106-108
                            linked[xa] |= xcc; linked[xc] |= xca;
                            ++n_links;
                        } while (false);
                    }
                    absorbed = __shfl_sync(0xffffffffu, absorbed, 0);
                    if (absorbed) {                                           // every matching after this one: test again
                        pending = __ballot_sync(0xffffffffu, key != 0ull) & (src == 31 ? 0u : ~((2u << src) - 1u));
                        break;
                    }
                }
                __syncwarp();                                                 // lane 0's state before the next tests
            }
        }
    }
    bsync();

    // ---- connected components in first-seen order, BFS by levels (:117-130) ----
    for (int h = tid; h < H; h += nt) flag[h] = 0;                               // reuse as "done"
    bsync();
    if (tid == 0) n_links_s = n_links;
    bsync();
    // Warp 0 walks the components: the order-dependent steps (queue, set insertions) stay on lane 0, the scan of the
    // link list for the links of the head being expanded is spread over the lanes - 32 links per step, matches
    // taken in link order - which is what made a 160-head frame spend 2 ms here on one lane.
    if (tid < 32) {
        const int n_lk = n_links_s;
        int n_out = 0;
        IntSet comp;
        for (int f = 0; f < n_seen; ++f) {
            const int v = first_seen[f];
            if (flag[v]) continue;                                           // uniform: every lane reads the same word
            if (lane == 0) {
                comp.init(tab_a, tab_b);
                comp.add(v);
                flag[v] = 1;
                queue[0] = v;
            }
            __syncwarp();
            int qb = 0, qe = 1, size = 1;
            while (qb < qe) {
                const int x = queue[qb++];
                for (int i0 = 0; i0 < n_lk; i0 += 32) {
                    const int i = i0 + lane;
                    int w = -1;
                    if (i < n_lk) {
                        const int la = link_a[2 * i], lc = link_a[2 * i + 1];
                        if (la == x) w = lc; else if (lc == x) w = la;
                        if (w >= 0 && flag[w]) w = -1;
                    }
                    unsigned bal = __ballot_sync(0xffffffffu, w >= 0);
                    while (bal) {                                            // a head is linked to x at most once
                        const int src = __ffs(bal) - 1;
                        bal &= bal - 1;
                        const int wv = __shfl_sync(0xffffffffu, w, src);
                        if (lane == 0) { flag[wv] = 1; comp.add(wv); queue[qe] = wv; }
                        ++qe; ++size;
                    }
                }
                __syncwarp();
            }
            if (size < p.min_views) continue;
            if (lane == 0) {
                int* person = p.person_heads + (size_t)(h0 + n_out) * p.v_sm;
                for (int s = 0; s < p.v_sm; ++s) person[s] = -1;
                for (int i = 0; i <= comp.mask; ++i)
                    if (comp.tab[i] >= 0) person[cam[comp.tab[i]]] = comp.tab[i];
            }
            ++n_out;
        }
        if (lane == 0) p.n_persons[b] = n_out;
    }
}

// flattens per-frame person slots into a dense person list with global skeleton ids per camera
__global__ void gather_persons_kernel(int n_frames, const int* __restrict__ head_off, const int* __restrict__ person_heads,
                                      const int* __restrict__ n_persons, const int* __restrict__ person_off,
                                      const int* __restrict__ sm_slot, int v_sm, int n_cameras,
                                      int* __restrict__ person_sk, int* __restrict__ person_frame)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_frames) return;
    const int h0 = head_off[b];
    const int np = n_persons[b];
    const int o = person_off[b];
    for (int q = 0; q < np; ++q) {
        const int* ph = person_heads + (size_t)(h0 + q) * v_sm;
        for (int c = 0; c < n_cameras; ++c) {
            const int slot = sm_slot[c];
            const int h = slot >= 0 ? ph[slot] : -1;
            person_sk[(size_t)(o + q) * n_cameras + c] = h >= 0 ? h0 + h : -1;
        }
        person_frame[o + q] = b;
    }
}

// single-CTA exclusive scan (n up to a few million): out[0..n] with out[n] = total
__global__ void __launch_bounds__(1024) exclusive_scan_kernel(const int* __restrict__ in, int n, int* __restrict__ out)
{
    __shared__ int part[1024];
    const int tid = threadIdx.x;
    const int per = (n + 1023) / 1024;
    const int beg = min(n, tid * per), end = min(n, beg + per);
    int s = 0;
    for (int i = beg; i < end; ++i) s += in[i];
    part[tid] = s;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        int v = tid >= d ? part[tid - d] : 0;
        __syncthreads();
        part[tid] += v;
        __syncthreads();
    }
    int run = tid ? part[tid - 1] : 0;
    for (int i = beg; i < end; ++i) { out[i] = run; run += in[i]; }
    if (tid == 1023) out[n] = part[1023];
}

// One rank's results as the fixed-size record of the final gather (sharding.py): word 0 = persons, then n_persons of
// every frame, the person list with batch-global skeleton ids, the joints as raw fp32 bits. The person count is read
// on the device (person_off[n_frames]), so nothing here waits for the host; padding words are never read back.
__global__ void __launch_bounds__(256) pack_record_kernel(
    int n_frames, int n_cameras, int n_out, const int* __restrict__ n_persons, const int* __restrict__ person_off,
    const int* __restrict__ person_sk, const float* __restrict__ joints, int ld_joints, int frames_cap, int persons_cap,
    int head_base, int* __restrict__ rec)
{
    const int P = min(person_off[n_frames], persons_cap);
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nthr = gridDim.x * blockDim.x;
    if (tid == 0) rec[0] = person_off[n_frames];
    for (int i = tid; i < n_frames; i += nthr) rec[1 + i] = n_persons[i];
    int* sk = rec + 1 + frames_cap;
    for (int i = tid; i < P * n_cameras; i += nthr) {
        const int v = person_sk[i];
        sk[i] = v >= 0 ? v + head_base : v;
    }
    float* jo = reinterpret_cast<float*>(sk + (size_t)persons_cap * n_cameras);
    if (joints)
        for (int i = tid; i < P * n_out; i += nthr) {
            const int r = i / n_out, c = i - r * n_out;
            jo[i] = joints[(size_t)r * ld_joints + c];
        }
}

}  // namespace b200pose

using namespace b200pose;

static int set_table_capacity(int max_heads) {
    // largest CPython set table reached while inserting max_heads distinct keys
    int mask = 7, fill = 0;
    for (int i = 0; i < max_heads; ++i) {
        ++fill;
        if (fill * 5 >= mask * 3) {
            int newsize = 8;
            while (newsize <= fill * 4) newsize <<= 1;
            mask = newsize - 1;
        }
    }
    return mask + 1;
}

static int cluster_launch(int32_t n_frames, const int32_t* head_off, const int32_t* node_off,
                          const int32_t* pairs, const int32_t* node_cam, const float* scores,
                          int32_t v_sm, double threshold, int32_t min_views,
                          int32_t max_heads_per_frame, int32_t max_enodes_per_frame,
                          int32_t* person_heads, int32_t* n_persons, int general, void* stream)
{
    B2_CHECK_ARG(head_off && node_off && pairs && node_cam && scores && person_heads && n_persons, "cluster: null pointer");
    B2_CHECK_ARG(v_sm >= 1 && v_sm <= B200POSE_MAX_CAMERAS, "cluster: v_sm out of range");
    if (n_frames == 0) return B200POSE_OK;
    ClusterParams p;
    p.head_off = head_off; p.node_off = node_off; p.pairs = pairs; p.node_cam = node_cam; p.scores = scores;
    p.v_sm = v_sm; p.threshold = threshold; p.min_views = min_views; p.person_heads = person_heads; p.n_persons = n_persons;
    p.general = general;
    p.max_heads = max_heads_per_frame < 1 ? 1 : max_heads_per_frame;
    int keys = 1;
    while (keys < max_enodes_per_frame) keys <<= 1;
    p.max_keys = keys;
    p.table_cap = set_table_capacity(p.max_heads);
    const size_t smem = (size_t)p.max_keys * 8 + (size_t)p.max_heads * 7 * 4 + (size_t)p.table_cap * 2 * 4;
    if (smem > 200 * 1024) {
        set_error("cluster: frame too large for the shared-memory plan (%zu bytes: %d heads, %d edge-nodes)", smem,
                  max_heads_per_frame, max_enodes_per_frame);
        return B200POSE_E_UNSUPPORTED;
    }
    if (p.max_keys > 4096) {
        B2_CHECK_CUDA(cudaFuncSetAttribute(cluster_kernel<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cluster_kernel<1024><<<n_frames, 1024, smem, (cudaStream_t)stream>>>(p);
    } else {
        B2_CHECK_CUDA(cudaFuncSetAttribute(cluster_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cluster_kernel<256><<<n_frames, p.max_keys > 1024 ? 256 : 32, smem, (cudaStream_t)stream>>>(p);
    }
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}

extern "C" __attribute__((visibility("default"))) int b200pose_cluster(int32_t n_frames, const int32_t* head_off, const int32_t* node_off,
                                const int32_t* pairs, const int32_t* node_cam, const float* scores,
                                int32_t v_sm, double threshold, int32_t min_views,
                                int32_t max_heads_per_frame, int32_t max_enodes_per_frame,
                                int32_t* person_heads, int32_t* n_persons, void* stream)
{
    return cluster_launch(n_frames, head_off, node_off, pairs, node_cam, scores, v_sm, threshold, min_views, max_heads_per_frame,
                          max_enodes_per_frame, person_heads, n_persons, 0, stream);
}

extern "C" __attribute__((visibility("default"))) int b200pose_cluster_pairs(int32_t n_graphs, const int32_t* head_off, const int32_t* node_off,
                                      const int32_t* pairs, const int32_t* node_cam, const float* scores,
                                      int32_t v_sm, double threshold, int32_t min_views,
                                      int32_t max_heads_per_graph, int32_t max_enodes_per_graph,
                                      int32_t* person_heads, int32_t* n_persons, void* stream)
{
    return cluster_launch(n_graphs, head_off, node_off, pairs, node_cam, scores, v_sm, threshold, min_views, max_heads_per_graph,
                          max_enodes_per_graph, person_heads, n_persons, 1, stream);
}

extern "C" __attribute__((visibility("default"))) int b200pose_gather_persons(int32_t n_frames, const int32_t* head_off, const int32_t* person_heads,
                                       const int32_t* n_persons, int32_t* person_off, int32_t scan,
                                       const int32_t* sk_cam, int32_t v_sm, const b200pose_cameras* cams,
                                       int32_t* person_sk, int32_t* person_frame, void* stream)
{
    (void)sk_cam;
    B2_CHECK_ARG(head_off && person_heads && n_persons && person_off && cams, "gather_persons: null pointer");
    if (n_frames == 0) return B200POSE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (scan) {
        exclusive_scan_kernel<<<1, 1024, 0, st>>>(n_persons, n_frames, person_off);
        B2_CHECK_LAUNCH();
    }
    if (person_sk) {
        B2_CHECK_ARG(person_frame, "gather_persons: person_frame missing");
        gather_persons_kernel<<<ceil_div(n_frames, 128), 128, 0, st>>>(n_frames, head_off, person_heads, n_persons, person_off,
                                                                       cams->sm_slot, v_sm, cams->n_cameras, person_sk, person_frame);
        B2_CHECK_LAUNCH();
    }
    return B200POSE_OK;
}

extern "C" __attribute__((visibility("default"))) int b200pose_pack_record(int32_t n_frames, int32_t n_cameras, int32_t n_out,
                                    const int32_t* n_persons, const int32_t* person_off, const int32_t* person_sk,
                                    const float* joints, int32_t ld_joints, int32_t frames_cap, int32_t persons_cap,
                                    int32_t head_base, int32_t* record, void* stream)
{
    B2_CHECK_ARG(n_persons && person_off && person_sk && record, "pack_record: null pointer");
    B2_CHECK_ARG(n_frames >= 0 && n_frames <= frames_cap && persons_cap >= 0 && n_cameras >= 1 && n_out >= 0, "pack_record: bad sizes");
    B2_CHECK_ARG(joints == nullptr || ld_joints >= n_out, "pack_record: ld_joints < n_out");
    const long long work = (long long)persons_cap * (n_out > n_cameras ? n_out : n_cameras);
    int blocks = (int)((work + 255) / 256);
    if (blocks < 1) blocks = 1;
    if (blocks > 592) blocks = 592;                 // 4 CTAs per SM: a copy of a few hundred KB
    pack_record_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(n_frames, n_cameras, n_out, n_persons, person_off, person_sk, joints,
                                                                   ld_joints, frames_cap, persons_cap, head_base, record);
    B2_CHECK_LAUNCH();
    return B200POSE_OK;
}
