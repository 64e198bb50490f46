// Frame-deduplicated replay: the opt-in layout of core/buffer/frame_replay.py for uint8 frame-stack fields [S, H, W].
//
// Replaces, for those fields, the duplicated ring rows of csrc/replay.cu (jorldy/core/buffer/replay_buffer.py:16-31 ring
// write, base.py:42-56 stack_transition, per_buffer.py:95-96 PER gather).  Each distinct frame is stored once in a pool
// frames[F, H*W] under a monotonically increasing int64 id (pool slot = id % F); a ring slot keeps the S ids of each of its
// stacks (ref[field][slot, S]) and the oldest of them (min_ref[slot]).
//
// Store = four launches, no host synchronisation:
//   hash    one CTA per incoming frame: an order-independent XOR of mixed 16-byte words.  Only a pre-filter: reuse is
//           decided by a full byte compare, so the hash can never make a stored stack differ from its input.
//   plan    one CTA per actor walks its rows in order (row t*N + r of the batch is actor r at step t).  Each of the K = nf*S
//           frames of a row is checked against the actor's history (its last 16 distinct frames, most recently used first):
//           the first candidate with an equal hash AND equal bytes (16-byte loads, block-wide AND) is reused and moved to the
//           front; otherwise the frame is the actor's next new frame.  Ids no longer in the pool are not candidates.
//   assign  exclusive scan of the per-actor new-frame counts -> ids (actor-major: actor r's j-th new frame gets
//           next_id + offs[r] + j), then the overflow check: neither a slot that stays live after this store (min_ref) nor
//           a row of this store (its reused ids) may reference an id the new frames overwrite (< next_id + total - F).
//           A violation sets the sticky ctl[3] flag.
//   commit  new frames -> pool (skipped while the flag is set), ref / min_ref rows, history codes -> ids.
// Integer atomics only set the flag; ids come from the scan, so the pool and the tables are identical run to run.
//
// Traffic per stored Atari transition (S = 4, 7 056 B frames, shapes only): the hash reads the 2 x 28 224 B input; steady
// state reuses 7 of its 8 frames and each reuse is one full compare (7 056 B candidate + 7 056 B input, L2-resident);
// candidates whose hash differs cost an 8 B shared-memory read.  Writes: one 7 056 B frame + 2 x 4 x 8 B ids + 8 B min_ref.
// The overflow check reads min_ref (8 B per slot) once per store.  Gather moves 2 x 28 224 B per sample, like replay.cu.
#include <limits.h>

#include "common.cuh"

namespace {

constexpr int HIST = 16;               // per-actor history length (>= S + n_step + 1 for every n-step window used here)
constexpr int MAX_FIELDS = 4;
constexpr long long EMPTY = LLONG_MIN; // unused history entry

struct Fields {
  const uint8_t* p[MAX_FIELDS];
};

__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}

// frame g of the batch: row g / K, frame k = g % K of that row (field k / S, stack position k % S)
__device__ __forceinline__ const uint4* batch_frame(const Fields& src, long long g, int K, int S, long long fb) {
  const long long row = g / K;
  const int k = (int)(g % K);
  return reinterpret_cast<const uint4*>(src.p[k / S] + (row * S + (k % S)) * fb);
}

__global__ void __launch_bounds__(128) frame_hash_kernel(Fields src, int K, int S, long long fb, uint64_t* __restrict__ hashes) {
  const long long g = blockIdx.x;
  const uint4* f = batch_frame(src, g, K, S, fb);
  uint64_t h = 0;
  for (long long q = threadIdx.x; q < fb / 16; q += blockDim.x) {
    const uint4 v = f[q];
    h ^= mix64((((uint64_t)v.y << 32) | v.x) ^ mix64((((uint64_t)v.w << 32) | v.z) + (uint64_t)q * 0x9e3779b97f4a7c15ull));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) h ^= __shfl_xor_sync(0xffffffffu, h, o);
  __shared__ uint64_t ws[4];
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = h;
  __syncthreads();
  if (threadIdx.x == 0) hashes[g] = ws[0] ^ ws[1] ^ ws[2] ^ ws[3];
}

// codes[g]: the pool id of a reused frame, or -(j + 1) for the actor's j-th new frame (newsrc[r * per + j] = g)
__global__ void __launch_bounds__(256) frame_plan_kernel(Fields src, int n_rows, int N, int K, int S, long long fb,
                                                         const uint8_t* __restrict__ frames, long long F,
                                                         const uint64_t* __restrict__ hashes, const long long* __restrict__ ctl,
                                                         long long* __restrict__ hist_id, uint64_t* __restrict__ hist_h,
                                                         long long* __restrict__ codes, long long* newsrc,
                                                         long long* __restrict__ counts) {
  const int r = blockIdx.x;
  const int T = n_rows / N;
  const long long per = (long long)T * K;
  __shared__ long long hid[HIST];
  __shared__ uint64_t hh[HIST];
  __shared__ long long s_count;
  if (threadIdx.x < HIST) {
    hid[threadIdx.x] = hist_id[(long long)r * HIST + threadIdx.x];
    hh[threadIdx.x] = hist_h[(long long)r * HIST + threadIdx.x];
  }
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  const long long lo = ctl[0] - F;                          // ids below this are no longer in the pool
  const long long nvec = fb / 16;
  for (int t = 0; t < T; ++t) {
    const long long row = (long long)t * N + r;
    for (int k = 0; k < K; ++k) {
      const long long g = row * K + k;
      const uint64_t h = hashes[g];
      const uint4* cur = batch_frame(src, g, K, S, fb);
      int found = -1;
      // every thread walks the same candidates (shared-memory values, block-uniform compare result)
      for (int w = 0; w < HIST; ++w) {
        const long long c = hid[w];
        if (c == EMPTY) break;                                 // the history is packed at the front
        if (hh[w] != h || (c >= 0 && c < lo)) continue;
        const uint4* cand = c >= 0 ? reinterpret_cast<const uint4*>(frames + (c % F) * fb)
                                   : batch_frame(src, newsrc[r * per + (-c - 1)], K, S, fb);
        int eq = 1;
        for (long long q = threadIdx.x; q < nvec; q += blockDim.x) {
          const uint4 a = cur[q], b = cand[q];
          eq &= (a.x == b.x) & (a.y == b.y) & (a.z == b.z) & (a.w == b.w);
        }
        if (__syncthreads_and(eq)) { found = w; break; }
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        long long code;
        uint64_t ch;
        int last;
        if (found >= 0) {
          code = hid[found]; ch = hh[found]; last = found;
        } else {
          const long long j = s_count++;
          newsrc[r * per + j] = g;
          code = -(j + 1); ch = h; last = HIST - 1;
        }
        for (int w = last; w > 0; --w) { hid[w] = hid[w - 1]; hh[w] = hh[w - 1]; }
        hid[0] = code; hh[0] = ch;
        codes[g] = code;
      }
      __syncthreads();
    }
  }
  if (threadIdx.x < HIST) {
    hist_id[(long long)r * HIST + threadIdx.x] = hid[threadIdx.x];
    hist_h[(long long)r * HIST + threadIdx.x] = hh[threadIdx.x];
  }
  if (threadIdx.x == 0) counts[r] = s_count;
}

// single CTA: offs = exclusive scan of counts; ctl = {next_id + total, next_id, total, flag | total > F}
__global__ void __launch_bounds__(1024) frame_assign_kernel(const long long* __restrict__ counts, int N, long long F,
                                                            long long* __restrict__ offs, long long* __restrict__ ctl) {
  __shared__ long long part[1024];
  const int tid = threadIdx.x;
  const int per = (N + blockDim.x - 1) / blockDim.x;
  const int b = min(N, tid * per), e = min(N, b + per);
  long long s = 0;
  for (int i = b; i < e; ++i) s += counts[i];
  part[tid] = s;
  __syncthreads();
  for (int o = 1; o < (int)blockDim.x; o <<= 1) {
    const long long v = tid >= o ? part[tid - o] : 0;
    __syncthreads();
    part[tid] += v;
    __syncthreads();
  }
  long long run = part[tid] - s;
  for (int i = b; i < e; ++i) { offs[i] = run; run += counts[i]; }
  if (tid == (int)blockDim.x - 1) {
    const long long total = part[tid], base = ctl[0];
    ctl[0] = base + total;
    ctl[1] = base;
    ctl[2] = total;
    if (total > F) ctl[3] = 1;                                 // one store would overwrite its own new frames
  }
}

// flags a reference to an id the new frames overwrite: from a slot outside the rows [start, start + nw) being rewritten
// (min_ref), or from a reused frame of this store (codes >= 0)
__global__ void frame_check_kernel(const long long* __restrict__ min_ref, long long cap, long long start, long long nw,
                                   const long long* __restrict__ codes, long long n_codes, long long F, long long* ctl) {
  const long long lo = ctl[1] + ctl[2] - F;
  int bad = 0;
  for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < cap + n_codes; s += (long long)gridDim.x * blockDim.x) {
    if (s >= cap) {
      const long long c = codes[s - cap];
      bad |= c >= 0 && c < lo;
      continue;
    }
    long long d = s - start;
    if (d < 0) d += cap;
    if (d >= nw) bad |= min_ref[s] < lo;
  }
  if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(reinterpret_cast<unsigned long long*>(ctl + 3), 1ull);
}

__global__ void __launch_bounds__(128) frame_commit_frames_kernel(Fields src, int K, int S, long long fb, uint8_t* __restrict__ frames,
                                                                  long long F, const long long* __restrict__ ctl,
                                                                  const long long* __restrict__ counts,
                                                                  const long long* __restrict__ offs,
                                                                  const long long* __restrict__ newsrc, long long per) {
  if (ctl[3]) return;                                          // overflow: keep the frames live slots still reference
  const int r = blockIdx.x;
  const long long first = ctl[1] + offs[r], cnt = counts[r];
  for (long long j = blockIdx.y; j < cnt; j += gridDim.y) {
    const uint4* s4 = batch_frame(src, newsrc[r * per + j], K, S, fb);
    uint4* d4 = reinterpret_cast<uint4*>(frames + ((first + j) % F) * fb);
    for (long long q = threadIdx.x; q < fb / 16; q += blockDim.x) d4[q] = s4[q];
  }
}

// threads [0, n_rows): ref / min_ref of the surviving rows; then N * HIST threads: history codes -> ids
__global__ void frame_commit_refs_kernel(const long long* __restrict__ codes, int n_rows, int N, int K, int S,
                                         const long long* __restrict__ ctl, const long long* __restrict__ offs,
                                         long long* __restrict__ ref, long long* __restrict__ min_ref, long long cap,
                                         long long start, long long keep_from, long long* __restrict__ hist_id) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long base = ctl[1];
  if (i < n_rows) {
    if (i < keep_from) return;
    const int r = (int)(i % N);
    const long long pos = (start + i) % cap;
    long long m = LLONG_MAX;
    for (int k = 0; k < K; ++k) {
      const long long c = codes[i * K + k];
      const long long id = c >= 0 ? c : base + offs[r] + (-c - 1);
      ref[((long long)(k / S) * cap + pos) * S + (k % S)] = id;
      m = min(m, id);
    }
    min_ref[pos] = m;
  } else if (i < n_rows + (long long)N * HIST) {
    const long long j = i - n_rows;
    const long long c = hist_id[j];
    if (c < 0 && c != EMPTY) hist_id[j] = base + offs[j / HIST] + (-c - 1);
  }
}

__global__ void __launch_bounds__(128) frame_gather_kernel(const uint8_t* __restrict__ frames, long long F, long long fb,
                                                           const long long* __restrict__ ref, int S,
                                                           const long long* __restrict__ idx, uint8_t* __restrict__ out) {
  const int s = blockIdx.x;
  const long long b = blockIdx.y;
  const long long id = ref[idx[b] * S + s];
  const uint4* s4 = reinterpret_cast<const uint4*>(frames + (id % F) * fb);
  uint4* d4 = reinterpret_cast<uint4*>(out + (b * S + s) * fb);
  for (long long q = threadIdx.x; q < fb / 16; q += blockDim.x) d4[q] = s4[q];
}

bool load_fields(const void* host_fields, int nf, Fields& f) {
  if (!host_fields || nf <= 0 || nf > MAX_FIELDS) return false;
  const uint8_t* const* p = static_cast<const uint8_t* const*>(host_fields);
  for (int i = 0; i < MAX_FIELDS; ++i) {
    f.p[i] = i < nf ? p[i] : nullptr;
    if (i < nf && (!p[i] || ((uintptr_t)p[i] & 15))) return false;
  }
  return true;
}

bool shapes_ok(int n, int N, int S, long long fb) {
  return n > 0 && N > 0 && n % N == 0 && S > 0 && fb > 0 && fb % 16 == 0;
}

}  // namespace

JB_API int jb_frame_plan(const void* host_fields, int nf, int n, int N, int S, long long frame_bytes, const uint8_t* frames,
                         int64_t F, uint64_t* hashes, const int64_t* ctl, int64_t* hist_id, uint64_t* hist_h, int64_t* codes,
                         int64_t* newsrc, int64_t* counts, void* stream) {
  Fields f;
  if (!load_fields(host_fields, nf, f) || !shapes_ok(n, N, S, frame_bytes) || !frames || F <= 0 || !hashes || !ctl ||
      !hist_id || !hist_h || !codes || !newsrc || !counts)
    return JB_ERR_INVALID;
  const int K = nf * S;
  cudaStream_t s = (cudaStream_t)stream;
  frame_hash_kernel<<<(unsigned)((long long)n * K), 128, 0, s>>>(f, K, S, frame_bytes, hashes);
  frame_plan_kernel<<<N, 256, 0, s>>>(f, n, N, K, S, frame_bytes, frames, F, hashes, (const long long*)ctl,
                                      (long long*)hist_id, hist_h, (long long*)codes, (long long*)newsrc, (long long*)counts);
  return jb_check_launch();
}

JB_API int jb_frame_assign(const int64_t* counts, int N, int64_t F, const int64_t* min_ref, int64_t capacity, int64_t start,
                           int64_t n, const int64_t* codes, int64_t n_codes, int64_t* offs, int64_t* ctl, void* stream) {
  if (!counts || N <= 0 || F <= 0 || !min_ref || capacity <= 0 || start < 0 || start >= capacity || n <= 0 || !codes ||
      n_codes <= 0 || !offs || !ctl)
    return JB_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  frame_assign_kernel<<<1, 1024, 0, s>>>((const long long*)counts, N, F, (long long*)offs, (long long*)ctl);
  const long long nw = n < capacity ? n : capacity;
  frame_check_kernel<<<jb_grid_for(capacity + n_codes, 256 * 8, 4), 256, 0, s>>>(
      (const long long*)min_ref, capacity, start, nw, (const long long*)codes, n_codes, F, (long long*)ctl);
  return jb_check_launch();
}

JB_API int jb_frame_commit(const void* host_fields, int nf, int n, int N, int S, long long frame_bytes, uint8_t* frames,
                           int64_t F, const int64_t* ctl, const int64_t* counts, const int64_t* offs, const int64_t* newsrc,
                           const int64_t* codes, int64_t* ref, int64_t* min_ref, int64_t capacity, int64_t start,
                           int64_t* hist_id, void* stream) {
  Fields f;
  if (!load_fields(host_fields, nf, f) || !shapes_ok(n, N, S, frame_bytes) || !frames || F <= 0 || !ctl || !counts ||
      !offs || !newsrc || !codes || !ref || !min_ref || capacity <= 0 || start < 0 || start >= capacity || !hist_id)
    return JB_ERR_INVALID;
  const int K = nf * S;
  const long long per = (long long)(n / N) * K;
  cudaStream_t s = (cudaStream_t)stream;
  dim3 grid(N, (unsigned)(per < 8 ? per : 8));
  frame_commit_frames_kernel<<<grid, 128, 0, s>>>(f, K, S, frame_bytes, frames, F, (const long long*)ctl,
                                                  (const long long*)counts, (const long long*)offs,
                                                  (const long long*)newsrc, per);
  const long long keep_from = n > capacity ? n - capacity : 0;
  const long long threads = (long long)n + (long long)N * HIST;
  frame_commit_refs_kernel<<<jb_div_up(threads, 256), 256, 0, s>>>(
      (const long long*)codes, n, N, K, S, (const long long*)ctl, (const long long*)offs, (long long*)ref,
      (long long*)min_ref, capacity, start, keep_from, (long long*)hist_id);
  return jb_check_launch();
}

JB_API int jb_frame_gather(const uint8_t* frames, int64_t F, long long frame_bytes, const int64_t* ref, int S,
                           const int64_t* idx, int B, uint8_t* out, void* stream) {
  if (!frames || F <= 0 || frame_bytes <= 0 || frame_bytes % 16 || !ref || S <= 0 || !idx || B <= 0 || B > 65535 || !out ||
      ((uintptr_t)out & 15))
    return JB_ERR_INVALID;
  frame_gather_kernel<<<dim3(S, B), 128, 0, (cudaStream_t)stream>>>(frames, F, frame_bytes, (const long long*)ref, S,
                                                                    (const long long*)idx, out);
  return jb_check_launch();
}
