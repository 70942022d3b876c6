// bow.cu -- bag-of-words pieces of the tracking fallback path (Tracking::TrackReferenceKeyFrame, src/Tracking.cc:858-904):
//   DBoW2::TemplatedVocabulary::transform(features, BowVector&, FeatureVector&, levelsup)   Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1140-1272
//       (Frame::ComputeBoW, src/Frame.cc:421-428, levelsup = 4): greedy descent of the k-ary tree by Hamming distance, first child wins ties;
//   ORBmatcher::SearchByBoW(KeyFrame*, Frame&, vector<MapPoint*>&)                           src/ORBmatcher.cc:159-290.
// The vocabulary lives on the device as flat arrays (the table the multi-GPU bench broadcasts once at start-up).
//   transform : one warp per descriptor, one lane per child, the arg-min over (distance, child order) by redux.sync.
//   SearchByBoW: one block per (key frame, frame) pair.  Both feature sets are sorted by (node id, feature index) -- the order of
//       DBoW2::FeatureVector (std::map<NodeId, vector<unsigned>>).  A frame feature belongs to exactly one node, so node buckets are
//       independent: each bucket is handled by one warp, key-frame features in order (the claims of earlier ones are visible), lanes
//       over the frame features of the bucket; best / second-best by two warp reductions.  Rotation histogram as in the other matchers.
// Integer work: bit-exact against the CPU restatement.
#include <cuda_runtime.h>

#include <stdexcept>
#include <string>
#include <cstdlib>
#include <cstdio>

#include <cstring>
#include <vector>

#include "host_call.h"
#include "sgs_common.h"

struct sgs_vocabulary {
    int device = 0, k = 0, L = 0, nnodes = 0;
    int32_t* d_first = nullptr; int32_t* d_count = nullptr; int32_t* d_children = nullptr; int32_t* d_word = nullptr;
    uint8_t* d_desc = nullptr; double* d_weight = nullptr;
};

namespace sgs {

constexpr int kBowThreads = 256;
constexpr int kBowThLow = 50, kBowHisto = 30;      // TH_LOW, HISTO_LENGTH (src/ORBmatcher.cc:37-39)

struct VocDev { const int32_t* first; const int32_t* count; const int32_t* children; const int32_t* word; const uint8_t* desc; const double* weight; int L; };

__device__ __forceinline__ int popc256v(const uint4& a0, const uint4& a1, const uint4& b0, const uint4& b1) {
    return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) + __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) +
           __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

__global__ void __launch_bounds__(256) bow_transform_kernel(const VocDev V, const uint8_t* __restrict__ desc, const int32_t* __restrict__ counts, int cap,
                                                            int levelsup, int32_t* __restrict__ word, double* __restrict__ weight, int32_t* __restrict__ node) {
    const int f = blockIdx.y, lane = threadIdx.x & 31;
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int n = counts ? min(counts[f], cap) : cap;
    if (i >= n) return;
    const int64_t o = (int64_t)f * cap + i;
    const uint4* d = reinterpret_cast<const uint4*>(desc + 32 * o);
    const uint4 d0 = __ldg(d), d1 = __ldg(d + 1);
    const int nid_level = V.L - levelsup;
    int cur = 0, level = 0, nid = 0;
    int nch = V.count[0];
    while (nch > 0) {
        ++level;
        const int first = V.first[cur];
        unsigned best = 0xffffffffu;
        for (int c0 = 0; c0 < nch; c0 += 32) {          // children in order; (distance << 12 | order) keeps the first of equal distances
            const int c = c0 + lane;
            if (c < nch) {
                const uint4* cd = reinterpret_cast<const uint4*>(V.desc + 32 * (int64_t)__ldg(V.children + first + c));
                best = min(best, ((unsigned)popc256v(d0, d1, __ldg(cd), __ldg(cd + 1)) << 12) | (unsigned)c);
            }
        }
        best = __reduce_min_sync(0xffffffffu, best);
        cur = __ldg(V.children + first + (int)(best & 0xfffu));
        if (level == nid_level) nid = cur;
        nch = V.count[cur];
    }
    if (lane == 0) { word[o] = V.word[cur]; weight[o] = V.weight[cur]; node[o] = nid; }
}

struct BowArgs {
    const int32_t* kf_node; const double* kf_weight; const uint8_t* kf_valid; const uint8_t* kf_desc; const float* kf_angle; const int32_t* kf_n; int kf_cap;
    const int32_t* f_node; const double* f_weight; const uint8_t* f_valid; const uint8_t* f_desc; const float* f_angle; const int32_t* f_n; int f_cap;
    float nnratio; int check_ori;
    int pair_mode;              // 1: SearchByBoW(KF1, KF2): strict < TH_LOW, second side needs map points, result indexed by the first side
                                // 2: SearchForTriangulation: no ratio test, epipole + epipolar-line gates, last of equal distances wins
    const uint8_t* kf_stereo; const uint8_t* f_stereo; const float* kf_xy; const float* f_xy; const int32_t* f_octave;
    const float* F12; const float* epipole; float sigma2[16], scale[16]; int only_stereo;
    int32_t* match_f; int32_t* nmatches;
    int kf_pow2, f_pow2;
};

__device__ void bow_bitonic(uint64_t* keys, int n_pow2) {         // ascending, n_pow2 a power of two, padding = all ones
    for (int k = 2; k <= n_pow2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n_pow2; i += blockDim.x) {
                const int p = i ^ j;
                if (p > i) {
                    const uint64_t a = keys[i], b = keys[p];
                    const bool up = (i & k) == 0;
                    if ((a > b) == up) { keys[i] = b; keys[p] = a; }
                }
            }
            __syncthreads();
        }
}

// keys: (node id << 32 | feature index)
__global__ void __launch_bounds__(kBowThreads) bow_search_kernel(const BowArgs A) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint64_t* kkey = reinterpret_cast<uint64_t*>(smem);            // [kf_pow2]
    uint64_t* fkey = kkey + A.kf_pow2;                              // [f_pow2]
    int32_t* run_start = reinterpret_cast<int32_t*>(fkey + A.f_pow2);   // [kf_pow2 + 1]
    int32_t* events = run_start + A.kf_pow2 + 1;                    // [max(kf_cap, f_cap)] (bin << 16 | index in the result array)
    uint8_t* taken = reinterpret_cast<uint8_t*>(events + max(A.kf_cap, A.f_cap));  // [f_cap]
    __shared__ int hist[kBowHisto];
    __shared__ int s_nk, s_nf, s_nruns, s_nevent, s_nmatch;
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nk_all = min(A.kf_n[f], A.kf_cap), nf_all = min(A.f_n[f], A.f_cap);
    const int64_t ko = (int64_t)f * A.kf_cap, fo = (int64_t)f * A.f_cap;
    if (tid == 0) { s_nk = 0; s_nf = 0; s_nruns = 0; s_nevent = 0; s_nmatch = 0; }
    if (tid < kBowHisto) hist[tid] = 0;
    for (int i = tid; i < A.kf_pow2; i += blockDim.x) {
        uint64_t key = ~0ull;
        if (i < nk_all && A.kf_weight[ko + i] > 0 && A.kf_valid[ko + i] && !(A.pair_mode == 2 && A.only_stereo && !A.kf_stereo[ko + i])) key = ((uint64_t)(uint32_t)A.kf_node[ko + i] << 32) | (uint32_t)i;      // invalid map points never act
        kkey[i] = key;
    }
    for (int j = tid; j < A.f_pow2; j += blockDim.x) {
        uint64_t key = ~0ull;
        if (j < nf_all && A.f_weight[fo + j] > 0 && (!A.f_valid || A.f_valid[fo + j]) && !(A.pair_mode == 2 && A.only_stereo && !A.f_stereo[fo + j])) key = ((uint64_t)(uint32_t)A.f_node[fo + j] << 32) | (uint32_t)j;
        fkey[j] = key;
    }
    const int64_t oo = A.pair_mode ? ko : fo;                      // the result is indexed by the first side in pair mode
    for (int j = tid; j < A.f_cap; j += blockDim.x) taken[j] = 0;
    for (int j = tid; j < (A.pair_mode ? A.kf_cap : A.f_cap); j += blockDim.x) A.match_f[oo + j] = -1;
    __syncthreads();
    bow_bitonic(kkey, A.kf_pow2);
    bow_bitonic(fkey, A.f_pow2);
    // number of live entries and the starts of the key-frame node runs
    for (int i = tid; i < A.kf_pow2; i += blockDim.x) {
        if (kkey[i] != ~0ull) {
            if (i + 1 == A.kf_pow2 || kkey[i + 1] == ~0ull) s_nk = i + 1;
            if (i == 0 || (kkey[i - 1] >> 32) != (kkey[i] >> 32)) run_start[atomicAdd(&s_nruns, 1)] = i;      // order of the runs does not matter
        }
    }
    for (int j = tid; j < A.f_pow2; j += blockDim.x)
        if (fkey[j] != ~0ull && (j + 1 == A.f_pow2 || fkey[j + 1] == ~0ull)) s_nf = j + 1;
    __syncthreads();
    const int nk = s_nk, nf = s_nf, nruns = s_nruns;
    const uint4* kdesc = reinterpret_cast<const uint4*>(A.kf_desc + 32 * ko);
    const uint4* fdesc = reinterpret_cast<const uint4*>(A.f_desc + 32 * fo);
    int nmatch = 0;
    for (int r = warp; r < nruns; r += kBowThreads / 32) {
        const int ks = run_start[r];
        const uint32_t nodeid = (uint32_t)(kkey[ks] >> 32);
        // the frame's bucket of this node: [lo, hi) in fkey
        int lo = 0, hi = nf;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if ((uint32_t)(fkey[mid] >> 32) < nodeid) lo = mid + 1; else hi = mid; }
        const int b0 = lo;
        hi = nf;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if ((uint32_t)(fkey[mid] >> 32) <= nodeid) lo = mid + 1; else hi = mid; }
        const int b1 = lo;
        if (b1 == b0) continue;
        for (int ki = ks; ki < nk && (uint32_t)(kkey[ki] >> 32) == nodeid; ++ki) {
            const int realK = (int)(uint32_t)kkey[ki];
            const uint4 k0 = __ldg(kdesc + 2 * realK), k1 = __ldg(kdesc + 2 * realK + 1);
            unsigned key1 = 0xffffffffu; int d2 = 256;              // local best (distance << 16 | bucket position), local second-best distance
            bool accept;
            unsigned K1;
            if (A.pair_mode == 2) {
                // SearchForTriangulation (:706-740): the best is the smallest distance <= TH_LOW among the candidates that pass the epipole and
                // epipolar-line gates; a later candidate replaces an earlier one of equal distance (dist > bestDist is the skip test)
                const float x1 = A.kf_xy[2 * (ko + realK)], y1 = A.kf_xy[2 * (ko + realK) + 1];
                const float* Fm = A.F12 + 9 * (int64_t)f;
                const float la = __fadd_rn(__fadd_rn(__fmul_rn(x1, Fm[0]), __fmul_rn(y1, Fm[3])), Fm[6]);        // CheckDistEpipolarLine (:140-157)
                const float lb = __fadd_rn(__fadd_rn(__fmul_rn(x1, Fm[1]), __fmul_rn(y1, Fm[4])), Fm[7]);
                const float lc = __fadd_rn(__fadd_rn(__fmul_rn(x1, Fm[2]), __fmul_rn(y1, Fm[5])), Fm[8]);
                const float den = __fadd_rn(__fmul_rn(la, la), __fmul_rn(lb, lb));
                const bool st1 = A.kf_stereo[ko + realK] != 0;
                const float ex = A.epipole[2 * f], ey = A.epipole[2 * f + 1];
                for (int p = b0 + lane; p < b1; p += 32) {
                    const int realF = (int)(uint32_t)fkey[p];
                    if (taken[realF]) continue;
                    const int dist = popc256v(k0, k1, __ldg(fdesc + 2 * realF), __ldg(fdesc + 2 * realF + 1));
                    if (dist > kBowThLow) continue;
                    const float x2 = A.f_xy[2 * (fo + realF)], y2 = A.f_xy[2 * (fo + realF) + 1];
                    const int oc = A.f_octave[fo + realF];
                    if (!st1 && !A.f_stereo[fo + realF]) {
                        const float dx = __fsub_rn(ex, x2), dy = __fsub_rn(ey, y2);
                        if (__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)) < __fmul_rn(100.f, A.scale[oc])) continue;
                    }
                    if (den == 0.f) continue;
                    const float num = __fadd_rn(__fadd_rn(__fmul_rn(la, x2), __fmul_rn(lb, y2)), lc);
                    const float dsqr = __fdiv_rn(__fmul_rn(num, num), den);
                    if (!((double)dsqr < 3.84 * (double)A.sigma2[oc])) continue;
                    key1 = min(key1, ((unsigned)dist << 16) | (unsigned)(0xffff - (p - b0)));
                }
                K1 = __reduce_min_sync(0xffffffffu, key1);
                accept = K1 != 0xffffffffu;
                if (accept) K1 = (K1 & 0xffff0000u) | (0xffffu - (K1 & 0xffffu));
            } else {
            for (int p = b0 + lane; p < b1; p += 32) {
                const int realF = (int)(uint32_t)fkey[p];
                if (taken[realF]) continue;                          // :214
                const int dist = popc256v(k0, k1, __ldg(fdesc + 2 * realF), __ldg(fdesc + 2 * realF + 1));
                const unsigned key = ((unsigned)dist << 16) | (unsigned)(p - b0);
                if (key < key1) { d2 = min(d2, (int)(key1 >> 16)); key1 = key; }
                else d2 = min(d2, dist);
            }
            K1 = __reduce_min_sync(0xffffffffu, key1);
            const int c2 = key1 == K1 ? d2 : min((int)(key1 >> 16), 256);
            const int best2 = __reduce_min_sync(0xffffffffu, c2 > 256 ? 256 : c2);
            const int best1 = K1 == 0xffffffffu ? 256 : (int)(K1 >> 16);
            accept = (A.pair_mode ? best1 < kBowThLow : best1 <= kBowThLow) && (float)best1 < __fmul_rn(A.nnratio, (float)best2);        // :237-240 / :599-601
            }
            if (accept) {
                const int realF = (int)(uint32_t)fkey[b0 + (int)(K1 & 0xffffu)];
                if (lane == 0) {
                    taken[realF] = 1;
                    const int slot = A.pair_mode ? realK : realF;
                    A.match_f[oo + slot] = A.pair_mode ? realF : realK;
                    if (A.check_ori) {
                        float rot = __fsub_rn(A.kf_angle[ko + realK], A.f_angle[fo + realF]);
                        if (rot < 0.f) rot = __fadd_rn(rot, 360.f);
                        int bin = (int)roundf(__fmul_rn(rot, (float)kBowHisto / 360.0f));
                        if (bin == kBowHisto) bin = 0;
                        atomicAdd(&hist[bin], 1);
                        events[atomicAdd(&s_nevent, 1)] = (bin << 16) | slot;
                    }
                    ++nmatch;
                }
                __syncwarp();
            }
        }
    }
    if (lane == 0 && nmatch) atomicAdd(&s_nmatch, nmatch);
    __syncthreads();
    if (A.check_ori) {
        // ComputeThreeMaxima (src/ORBmatcher.cc:1603-1645) on the bin counts, then drop the matches outside the three main bins
        __shared__ int s_i1, s_i2, s_i3;
        if (tid == 0) {
            int max1 = 0, max2 = 0, max3 = 0, i1 = -1, i2 = -1, i3 = -1;
            for (int i = 0; i < kBowHisto; ++i) {
                const int s = hist[i];
                if (s > max1) { max3 = max2; max2 = max1; max1 = s; i3 = i2; i2 = i1; i1 = i; }
                else if (s > max2) { max3 = max2; max2 = s; i3 = i2; i2 = i; }
                else if (s > max3) { max3 = s; i3 = i; }
            }
            if ((float)max2 < __fmul_rn(0.1f, (float)max1)) { i2 = -1; i3 = -1; }
            else if ((float)max3 < __fmul_rn(0.1f, (float)max1)) i3 = -1;
            s_i1 = i1; s_i2 = i2; s_i3 = i3;
        }
        __syncthreads();
        int removed = 0;
        for (int e = tid; e < s_nevent; e += blockDim.x) {
            const int bin = events[e] >> 16, j = events[e] & 0xffff;
            if (bin != s_i1 && bin != s_i2 && bin != s_i3) { A.match_f[oo + j] = -1; ++removed; }
        }
        if (removed) atomicSub(&s_nmatch, removed);
        __syncthreads();
    }
    if (tid == 0) A.nmatches[f] = s_nmatch;
}

static int pow2_ge(int n) { int p = 1; while (p < n) p <<= 1; return p; }

}  // namespace sgs

using namespace sgs;

extern "C" {

SGS_API void sgs_vocabulary_destroy(sgs_vocabulary* v) {
    if (!v) return;
    cudaSetDevice(v->device);
    cudaFree(v->d_first); cudaFree(v->d_count); cudaFree(v->d_children); cudaFree(v->d_word); cudaFree(v->d_desc); cudaFree(v->d_weight);
    delete v;
}

static int vocabulary_create_impl(int device, int k, int L, int nnodes, const int32_t* parent, const uint8_t* node_desc, bool desc_on_device,
                                  const double* node_weight, sgs_vocabulary** out) {
    if (!out || !parent || !node_desc || !node_weight || nnodes < 2 || k < 2 || L < 1) { set_error("sgs_vocabulary_create: bad argument"); return SGS_ERR_INVALID; }
    *out = nullptr;
    std::vector<int32_t> count(nnodes, 0), first(nnodes, 0), children(nnodes - 1), word(nnodes, -1), fill(nnodes, 0);
    for (int i = 1; i < nnodes; ++i) {
        if (parent[i] < 0 || parent[i] >= i) { set_error("sgs_vocabulary_create: parent[%d] = %d must name an earlier node", i, parent[i]); return SGS_ERR_INVALID; }
        count[parent[i]]++;
    }
    if (count[0] == 0) { set_error("sgs_vocabulary_create: the root has no children"); return SGS_ERR_INVALID; }
    int acc = 0;
    for (int i = 0; i < nnodes; ++i) { first[i] = acc; acc += count[i]; if (count[i] > 4096) { set_error("sgs_vocabulary_create: more than 4096 children"); return SGS_ERR_UNSUPPORTED; } }
    for (int i = 1; i < nnodes; ++i) children[first[parent[i]] + fill[parent[i]]++] = i;      // children in node-id order, as DBoW2 appends them while loading
    int w = 0;
    for (int i = 1; i < nnodes; ++i) if (count[i] == 0) word[i] = w++;
    SGS_CUDA_TRY(cudaSetDevice(device));
    sgs_vocabulary* v = new sgs_vocabulary();
    v->device = device; v->k = k; v->L = L; v->nnodes = nnodes;
    cudaError_t e = cudaMalloc(&v->d_first, 4 * (size_t)nnodes);
    if (e == cudaSuccess) e = cudaMalloc(&v->d_count, 4 * (size_t)nnodes);
    if (e == cudaSuccess) e = cudaMalloc(&v->d_children, 4 * (size_t)nnodes);
    if (e == cudaSuccess) e = cudaMalloc(&v->d_word, 4 * (size_t)nnodes);
    if (e == cudaSuccess) e = cudaMalloc(&v->d_desc, 32 * (size_t)nnodes);
    if (e == cudaSuccess) e = cudaMalloc(&v->d_weight, 8 * (size_t)nnodes);
    if (e == cudaSuccess) e = cudaMemcpy(v->d_first, first.data(), 4 * (size_t)nnodes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->d_count, count.data(), 4 * (size_t)nnodes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->d_children, children.data(), 4 * (size_t)(nnodes - 1), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->d_word, word.data(), 4 * (size_t)nnodes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->d_desc, node_desc, 32 * (size_t)nnodes, desc_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->d_weight, node_weight, 8 * (size_t)nnodes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { set_error("sgs_vocabulary_create: %s", cudaGetErrorString(e)); sgs_vocabulary_destroy(v); return SGS_ERR_CUDA; }
    *out = v;
    return SGS_OK;
}

SGS_API int sgs_vocabulary_create(int device, int k, int L, int nnodes, const int32_t* parent, const uint8_t* node_desc, const double* node_weight,
                                  sgs_vocabulary** out) {
    return vocabulary_create_impl(device, k, L, nnodes, parent, node_desc, false, node_weight, out);
}
// node descriptors already on the device (the buffer an ncclBroadcast just filled): consumed in place, no bounce through the host
SGS_API int sgs_vocabulary_create_device(int device, int k, int L, int nnodes, const int32_t* parent, const uint8_t* d_node_desc, const double* node_weight,
                                         sgs_vocabulary** out) {
    return vocabulary_create_impl(device, k, L, nnodes, parent, d_node_desc, true, node_weight, out);
}

// ---- vocabulary files: ORBVocabulary::loadFromTextFile / loadFromBinaryFile (Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1351-1420, :1467-1508).
// Text: first line "k L scoring weighting", then one line per node in node-id order (the root is implicit): "parent isLeaf d0 ... d31 weight".
// Binary: uint32 nb_nodes (root included), uint32 size_node (= 41), int k, int L, int scoring, int weighting, then nb_nodes - 1 records
// { int32 parent; uint8 descriptor[32]; float weight; uint8 is_leaf }.  src/System.cc:69-73 picks the text reader for a ".txt" suffix.
// Blank lines of a text file are skipped (the reference's eof() loop turns a trailing newline into one undefined extra node).
namespace {
struct VocFile { int k = 0, L = 0; std::vector<int32_t> parent; std::vector<uint8_t> desc, leaf; std::vector<double> weight; };

int parse_vocabulary_file(const char* path, VocFile& V) {
    const std::string p(path);
    const bool text = p.size() >= 4 && p.compare(p.size() - 4, 4, ".txt") == 0;
    FILE* f = std::fopen(path, text ? "r" : "rb");
    if (!f) { set_error("vocabulary: cannot open %s", path); return SGS_ERR_INVALID; }
    struct Closer { FILE* f; ~Closer() { std::fclose(f); } } closer{f};
    V.parent.assign(1, -1); V.desc.assign(32, 0); V.leaf.assign(1, 0); V.weight.assign(1, 0.0);       // node 0 = root
    if (text) {
        int n1 = 0, n2 = 0;
        if (std::fscanf(f, "%d %d %d %d", &V.k, &V.L, &n1, &n2) != 4 || V.k < 0 || V.k > 20 || V.L < 1 || V.L > 10 || n1 < 0 || n1 > 5 || n2 < 0 || n2 > 3) {
            set_error("vocabulary: %s is not a DBoW2 text vocabulary", path); return SGS_ERR_INVALID; }
        std::vector<char> line(1 << 12);
        if (!std::fgets(line.data(), (int)line.size(), f)) return SGS_OK;            // rest of the header line
        while (std::fgets(line.data(), (int)line.size(), f)) {
            char* c = line.data();
            while (*c == ' ' || *c == '\t') ++c;
            if (*c == '\n' || *c == '\r' || *c == 0) continue;
            char* e = nullptr;
            const long pid = std::strtol(c, &e, 10); c = e;
            const long isleaf = std::strtol(c, &e, 10); c = e;
            const size_t nid = V.parent.size();
            if (pid < 0 || (size_t)pid >= nid) { set_error("vocabulary: %s: node %zu names parent %ld", path, nid, pid); return SGS_ERR_INVALID; }
            V.parent.push_back((int32_t)pid); V.leaf.push_back(isleaf > 0 ? 1 : 0);
            for (int i = 0; i < 32; ++i) { const long v = std::strtol(c, &e, 10); if (e == c) { set_error("vocabulary: %s: node %zu has a short descriptor", path, nid); return SGS_ERR_INVALID; } c = e; V.desc.push_back((uint8_t)v); }
            V.weight.push_back(std::strtod(c, &e));
        }
    } else {
        uint32_t nb = 0, sz = 0; int32_t hdr[4];
        if (std::fread(&nb, 4, 1, f) != 1 || std::fread(&sz, 4, 1, f) != 1 || std::fread(hdr, 4, 4, f) != 4 || sz != 41 || hdr[0] < 2 || hdr[0] > 20 || hdr[1] < 1 || hdr[1] > 10) {
            set_error("vocabulary: %s is not a DBoW2 binary vocabulary (41-byte nodes)", path); return SGS_ERR_INVALID; }
        V.k = hdr[0]; V.L = hdr[1];
        // saveToBinaryFile (:1514-1535) writes nb_nodes = m_nodes.size() -- the root INCLUDED -- and then records for nodes 1 .. nb_nodes-1.
        // (loadFromBinaryFile's eof() loop additionally re-reads the last record into a phantom node nb_nodes; it duplicates the last child of its
        // parent, which a strict '<' descent can never select, so it is not materialised here.)
        if (nb < 2) { set_error("vocabulary: %s holds no nodes", path); return SGS_ERR_INVALID; }
        nb -= 1;
        long here = std::ftell(f), end = -1;
        if (here >= 0 && std::fseek(f, 0, SEEK_END) == 0) { end = std::ftell(f); std::fseek(f, here, SEEK_SET); }
        if (here < 0 || end < 0 || (uint64_t)(end - here) < (uint64_t)nb * 41) { set_error("vocabulary: %s is truncated", path); return SGS_ERR_INVALID; }   // before allocating
        std::vector<uint8_t> buf((size_t)nb * 41);
        if (std::fread(buf.data(), 41, nb, f) != nb) { set_error("vocabulary: %s is truncated", path); return SGS_ERR_INVALID; }
        V.parent.reserve(nb + 1); V.desc.reserve(32 * ((size_t)nb + 1)); V.leaf.reserve(nb + 1); V.weight.reserve(nb + 1);
        for (uint32_t i = 0; i < nb; ++i) {
            const uint8_t* r = buf.data() + (size_t)i * 41;
            int32_t pid; float w;
            std::memcpy(&pid, r, 4); std::memcpy(&w, r + 36, 4);
            if (pid < 0 || (uint32_t)pid > i) { set_error("vocabulary: %s: node %u names parent %d", path, i + 1, pid); return SGS_ERR_INVALID; }
            V.parent.push_back(pid); V.desc.insert(V.desc.end(), r + 4, r + 36); V.weight.push_back((double)w); V.leaf.push_back(r[40] ? 1 : 0);
        }
    }
    if (V.parent.size() < 2) { set_error("vocabulary: %s holds no nodes", path); return SGS_ERR_INVALID; }
    return SGS_OK;
}
}  // namespace

SGS_API int sgs_vocabulary_parse_file(const char* path, int* k, int* L, int* nnodes, int32_t* parent, uint8_t* node_desc, double* node_weight, uint8_t* is_leaf,
                                      int cap) {
    if (!path || !nnodes) { set_error("sgs_vocabulary_parse_file: bad argument"); return SGS_ERR_INVALID; }
    VocFile V;
    int rc = SGS_OK;
    try { rc = parse_vocabulary_file(path, V); } catch (const std::exception& ex) { set_error("sgs_vocabulary_parse_file: %s while reading %s", ex.what(), path); return SGS_ERR_INVALID; }
    if (rc != SGS_OK) return rc;
    const int n = (int)V.parent.size();
    if (k) *k = V.k;
    if (L) *L = V.L;
    *nnodes = n;
    if (!parent && !node_desc && !node_weight && !is_leaf) return SGS_OK;                     // size query
    if (cap < n) { set_error("sgs_vocabulary_parse_file: %d nodes, capacity %d", n, cap); return SGS_ERR_CAPACITY; }
    if (parent) std::memcpy(parent, V.parent.data(), 4 * (size_t)n);
    if (node_desc) std::memcpy(node_desc, V.desc.data(), 32 * (size_t)n);
    if (node_weight) std::memcpy(node_weight, V.weight.data(), 8 * (size_t)n);
    if (is_leaf) std::memcpy(is_leaf, V.leaf.data(), (size_t)n);
    return SGS_OK;
}

SGS_API int sgs_vocabulary_load(const char* path, int device, sgs_vocabulary** out) {
    if (!path || !out) { set_error("sgs_vocabulary_load: bad argument"); return SGS_ERR_INVALID; }
    *out = nullptr;
    VocFile V;
    int rc = SGS_OK;
    try { rc = parse_vocabulary_file(path, V); } catch (const std::exception& ex) { set_error("sgs_vocabulary_load: %s while reading %s", ex.what(), path); return SGS_ERR_INVALID; }
    if (rc != SGS_OK) return rc;
    const int n = (int)V.parent.size();
    std::vector<int> nchild(n, 0);
    for (int i = 1; i < n; ++i) nchild[V.parent[i]]++;
    for (int i = 1; i < n; ++i)
        if ((nchild[i] == 0) != (V.leaf[i] != 0)) { set_error("sgs_vocabulary_load: %s: node %d is flagged %s but has %d children", path, i, V.leaf[i] ? "leaf" : "inner", nchild[i]); return SGS_ERR_UNSUPPORTED; }
    return sgs_vocabulary_create(device, V.k, V.L, n, V.parent.data(), V.desc.data(), V.weight.data(), out);
}

SGS_API int sgs_bow_transform_batch_device(const sgs_vocabulary* v, const uint8_t* d_desc, const int32_t* d_counts, int cap, int nframes, int levelsup,
                                           int32_t* d_word, double* d_weight, int32_t* d_node, void* stream) {
    if (!v || !d_desc || !d_word || !d_weight || !d_node || cap < 1 || nframes < 1) { set_error("sgs_bow_transform_batch_device: bad argument"); return SGS_ERR_INVALID; }
    VocDev V{v->d_first, v->d_count, v->d_children, v->d_word, v->d_desc, v->d_weight, v->L};
    dim3 grid((cap + 7) / 8, nframes);
    bow_transform_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(V, d_desc, d_counts, cap, levelsup, d_word, d_weight, d_node);
    SGS_CUDA_TRY(cudaGetLastError());
    return SGS_OK;
}

SGS_API int sgs_match_bow_batch_device(const sgs_bow_batch* a, int nframes, void* stream) {
    if (!a || !a->kf_node || !a->kf_weight || !a->kf_valid || !a->kf_desc || !a->kf_angle || !a->kf_n || !a->f_node || !a->f_weight || !a->f_desc || !a->f_angle ||
        !a->f_n || !a->match_f || !a->nmatches || nframes < 1) { set_error("sgs_match_bow_batch_device: bad argument"); return SGS_ERR_INVALID; }
    if (a->kf_cap < 1 || a->f_cap < 1 || a->kf_cap > 8192 || a->f_cap > 8192) { set_error("sgs_match_bow_batch_device: at most 8192 features per frame"); return SGS_ERR_UNSUPPORTED; }
    BowArgs A;
    A.kf_node = a->kf_node; A.kf_weight = a->kf_weight; A.kf_valid = a->kf_valid; A.kf_desc = a->kf_desc; A.kf_angle = a->kf_angle; A.kf_n = a->kf_n; A.kf_cap = a->kf_cap;
    A.f_node = a->f_node; A.f_weight = a->f_weight; A.f_valid = a->f_valid; A.pair_mode = a->keyframe_pair; A.f_desc = a->f_desc;
    A.kf_stereo = a->kf_stereo; A.f_stereo = a->f_stereo; A.kf_xy = a->kf_xy; A.f_xy = a->f_xy; A.f_octave = a->f_octave; A.F12 = a->F12; A.epipole = a->epipole;
    A.only_stereo = a->only_stereo;
    for (int l = 0; l < 16; ++l) { A.sigma2[l] = a->level_sigma2[l]; A.scale[l] = a->scale_factors[l]; }
    if (a->keyframe_pair < 0 || a->keyframe_pair > 2) { set_error("sgs_match_bow_batch_device: keyframe_pair must be 0, 1 or 2"); return SGS_ERR_INVALID; }
    if (a->keyframe_pair == 2 && (!a->kf_stereo || !a->f_stereo || !a->kf_xy || !a->f_xy || !a->f_octave || !a->F12 || !a->epipole || !a->f_valid)) {
        set_error("sgs_match_bow_batch_device: triangulation mode needs positions, octaves, stereo flags, F12 and the epipole"); return SGS_ERR_INVALID;
    } A.f_angle = a->f_angle; A.f_n = a->f_n; A.f_cap = a->f_cap;
    A.nnratio = a->nnratio; A.check_ori = a->check_orientation; A.match_f = a->match_f; A.nmatches = a->nmatches;
    A.kf_pow2 = pow2_ge(a->kf_cap); A.f_pow2 = pow2_ge(a->f_cap);
    const size_t smem = 8 * (size_t)A.kf_pow2 + 8 * (size_t)A.f_pow2 + 4 * (size_t)(A.kf_pow2 + 1) + 4 * (size_t)(a->kf_cap > a->f_cap ? a->kf_cap : a->f_cap) + (size_t)A.f_cap + 16;
    if (smem > 40 * 1024)      // per device and cheap: set whenever the default 48 KB would not do
        SGS_CUDA_TRY(cudaFuncSetAttribute(bow_search_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    bow_search_kernel<<<nframes, kBowThreads, smem, (cudaStream_t)stream>>>(A);
    SGS_CUDA_TRY(cudaGetLastError());
    return SGS_OK;
}

// host-pointer variants for one (key frame, frame) pair / one descriptor set
SGS_API int sgs_bow_transform(const sgs_vocabulary* v, const uint8_t* desc, int n, int levelsup, int32_t* word, double* weight, int32_t* node) {
    if (!v || n < 0 || (n > 0 && (!desc || !word || !weight || !node))) { set_error("sgs_bow_transform: bad argument"); return SGS_ERR_INVALID; }
    if (n == 0) return SGS_OK;
    SGS_CUDA_TRY(cudaSetDevice(v->device));
    HostCall c("sgs_bow_transform");
    const uint8_t* d_desc; int32_t *d_word, *d_node; double* d_weight;
    c.in(&d_desc, desc, 32 * (size_t)n); c.out(&d_word, word, n); c.out(&d_weight, weight, n); c.out(&d_node, node, n);
    if (int rc = c.upload()) return rc;
    if (int rc = sgs_bow_transform_batch_device(v, d_desc, nullptr, n, 1, levelsup, d_word, d_weight, d_node, nullptr)) return rc;
    return c.download();
}

SGS_API int sgs_match_bow(int nkf, const int32_t* kf_node, const double* kf_weight, const uint8_t* kf_valid, const uint8_t* kf_desc, const float* kf_angle,
                          int nf, const int32_t* f_node, const double* f_weight, const uint8_t* f_desc, const float* f_angle, float nnratio,
                          int check_orientation, int32_t* match_f, int* nmatches, int device) {
    if (!nmatches || nkf < 0 || nf < 0) { set_error("sgs_match_bow: bad argument"); return SGS_ERR_INVALID; }
    *nmatches = 0;
    if (nf > 0 && match_f) for (int j = 0; j < nf; ++j) match_f[j] = -1;
    if (nkf == 0 || nf == 0) return SGS_OK;
    if (!kf_node || !kf_weight || !kf_valid || !kf_desc || !kf_angle || !f_node || !f_weight || !f_desc || !f_angle || !match_f) { set_error("sgs_match_bow: NULL array"); return SGS_ERR_INVALID; }
    SGS_CUDA_TRY(cudaSetDevice(device));
    HostCall c("sgs_match_bow");
    sgs_bow_batch b;
    std::memset(&b, 0, sizeof b);
    c.in(&b.kf_node, kf_node, nkf); c.in(&b.kf_weight, kf_weight, nkf); c.in(&b.kf_valid, kf_valid, nkf); c.in(&b.kf_desc, kf_desc, 32 * (size_t)nkf);
    c.in(&b.kf_angle, kf_angle, nkf); c.in(&b.kf_n, &nkf, 1);
    c.in(&b.f_node, f_node, nf); c.in(&b.f_weight, f_weight, nf); c.in(&b.f_desc, f_desc, 32 * (size_t)nf); c.in(&b.f_angle, f_angle, nf); c.in(&b.f_n, &nf, 1);
    c.out(&b.match_f, match_f, nf); c.out(&b.nmatches, nmatches, 1);
    b.kf_cap = nkf; b.f_cap = nf; b.nnratio = nnratio; b.check_orientation = check_orientation;
    if (int rc = c.upload()) return rc;
    if (int rc = sgs_match_bow_batch_device(&b, 1, nullptr)) return rc;
    return c.download();
}

}  // extern "C"
