// fq_utf8.cuh — Utf8 columns on the device: bytewise comparison, dictionary encoding and gathering strings by index.
//
// Dictionary encoding turns a string column into UInt32 codes over a SORTED dictionary of its distinct valid strings, so
// that code order is string order and every string comparison, GROUP BY, ORDER BY and min/max runs as an integer one:
//   1. fq_dict_insert: one thread per valid row hashes its bytes and finds or claims its slot in an open-addressing table in
//      HBM.  An entry is (upper 32 bits of the 64-bit hash, representative row) in one word, so the claim (one 64-bit CAS)
//      also publishes it.  A hash match is confirmed by comparing the bytes with the representative row's.
//   2. fq_dict_flag + an exclusive scan (sort_scan) + fq_dict_compact: occupied slots -> dense distinct ids and the list of
//      representative rows.
//   3. fq_dict_chunk: big-endian 8-byte chunks (zero-padded) and the length of every distinct string; sorted LSD with the
//      radix sort of fq_sort.cuh (length, then chunk K-1 down to chunk 0) they give exact bytewise order, embedded NUL
//      bytes and prefixes included: a shorter string whose bytes match is padded with zeros and loses on the length.
//   4. fq_dict_rank + fq_dict_codes: rank[id] = position in sorted order, codes[row] = rank[id of the row's slot].
// fq_utf8_lens / fq_utf8_gather_bytes gather strings by row index (the sorted dictionary from the representative rows, and
// result columns from codes); fq_utf8_bounds_kernel finds a literal's (lower, upper) bound in a sorted dictionary.
#pragma once

#define FQ_DICT_EMPTY 0xFFFFFFFFFFFFFFFFull   // hash32 = row = 0xFFFFFFFF cannot occur: rows are fewer than 2^32 - 1

// bytewise order, shorter string first on a common prefix (Rust str / arrow)
__device__ __forceinline__ int fq_utf8_cmp(const unsigned char *a, fq_u32 la, const unsigned char *b, fq_u32 lb) {
  const fq_u32 n = la < lb ? la : lb;
  for (fq_u32 i = 0; i < n; i++) {
    const int d = (int)a[i] - (int)b[i];
    if (d) return d;
  }
  return la < lb ? -1 : (la > lb ? 1 : 0);
}

__device__ __forceinline__ fq_u64 fq_utf8_hash(const unsigned char *p, fq_u32 n) {
  fq_u64 h = 0x9E3779B97F4A7C15ull ^ n;
  fq_u32 i = 0;
  for (; i + 8 <= n; i += 8) {
    fq_u64 w = 0;
#pragma unroll
    for (int b = 0; b < 8; b++) w |= (fq_u64)p[i + b] << (8 * b);
    h = (h ^ w) * 0xFF51AFD7ED558CCDull;
    h ^= h >> 32;
  }
  fq_u64 w = 0;
  for (int b = 0; i < n; i++, b++) w |= (fq_u64)p[i] << (8 * b);
  h = (h ^ w) * 0xC4CEB9FE1A85EC53ull;
  h ^= h >> 29;
  h *= 0xFF51AFD7ED558CCDull;
  h ^= h >> 32;
  return h;
}

__global__ void __launch_bounds__(256) fq_dict_clear(unsigned long long *table, fq_u64 cap) {
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (fq_u64)gridDim.x * blockDim.x) table[i] = FQ_DICT_EMPTY;
}

// slot_of[row] = the table slot of the row's string (NULL rows: untouched)
__global__ void __launch_bounds__(256) fq_dict_insert(const int *off, const unsigned char *data, const fq_u8 *valid, fq_u64 n,
                                                      unsigned long long *table, fq_u64 mask, fq_u32 *slot_of) {
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (fq_u64)gridDim.x * blockDim.x) {
    if (valid && !valid[i]) continue;
    const unsigned char *s = data + off[i];
    const fq_u32 len = (fq_u32)(off[i + 1] - off[i]);
    const fq_u64 h = fq_utf8_hash(s, len);
    const fq_u64 tag = h >> 32;
    const unsigned long long mine = (tag << 32) | i;
    fq_u64 slot = h & mask;
    for (;;) {
      unsigned long long e = *(volatile unsigned long long *)(table + slot);   // look before any atomic
      if (e == FQ_DICT_EMPTY) {
        e = atomicCAS(table + slot, FQ_DICT_EMPTY, mine);
        if (e == FQ_DICT_EMPTY) break;   // claimed: this row represents the string
      }
      if ((e >> 32) == tag) {
        const fq_u32 r = (fq_u32)e;
        const fq_u32 lr = (fq_u32)(off[r + 1] - off[r]);
        if (lr == len && fq_utf8_cmp(data + off[r], lr, s, len) == 0) break;
      }
      slot = (slot + 1) & mask;
    }
    slot_of[i] = (fq_u32)slot;
  }
}

__global__ void __launch_bounds__(256) fq_dict_flag(const unsigned long long *table, fq_u64 cap, fq_u32 *ids) {
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (fq_u64)gridDim.x * blockDim.x)
    ids[i] = table[i] != FQ_DICT_EMPTY ? 1u : 0u;
}

// after the exclusive scan of the flags: rep[id] = representative row, len[id] = its length; max_len folded by atomicMax
__global__ void __launch_bounds__(256) fq_dict_compact(const unsigned long long *table, fq_u64 cap, const fq_u32 *ids, const int *off,
                                                       fq_u32 *rep, fq_u32 *len, fq_u32 *max_len) {
  fq_u32 m = 0;
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (fq_u64)gridDim.x * blockDim.x) {
    const unsigned long long e = table[i];
    if (e == FQ_DICT_EMPTY) continue;
    const fq_u32 r = (fq_u32)e, l = (fq_u32)(off[r + 1] - off[r]);
    rep[ids[i]] = r;
    len[ids[i]] = l;
    m = l > m ? l : m;
  }
  for (int o = 16; o > 0; o >>= 1) {
    const fq_u32 x = __shfl_xor_sync(0xffffffffu, m, o);
    m = x > m ? x : m;
  }
  if ((threadIdx.x & 31) == 0 && m) atomicMax(max_len, m);
}

// chunk[id] = bytes [8j, 8j + 8) of distinct string id, big-endian, zero-padded
__global__ void __launch_bounds__(256) fq_dict_chunk(const int *off, const unsigned char *data, const fq_u32 *rep, fq_u64 d, fq_u32 j,
                                                     fq_u64 *chunk) {
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i < d; i += (fq_u64)gridDim.x * blockDim.x) {
    const fq_u32 r = rep[i];
    const unsigned char *s = data + off[r];
    const fq_u32 len = (fq_u32)(off[r + 1] - off[r]);
    fq_u64 w = 0;
#pragma unroll
    for (int b = 0; b < 8; b++) {
      const fq_u32 at = 8 * j + b;
      w = (w << 8) | (at < len ? s[at] : 0);
    }
    chunk[i] = w;
  }
}

// sorted[r] = distinct id at sorted position r -> rank[id] = r and rows[r] = its representative row
__global__ void __launch_bounds__(256) fq_dict_rank(const fq_u32 *sorted, fq_u64 d, const fq_u32 *rep, fq_u32 *rank, fq_u32 *rows) {
  for (fq_u64 r = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; r < d; r += (fq_u64)gridDim.x * blockDim.x) {
    const fq_u32 id = sorted[r];
    rank[id] = (fq_u32)r;
    rows[r] = rep[id];
  }
}

// codes[row] = rank of the row's string; NULL rows get 0 (their validity says NULL)
__global__ void __launch_bounds__(256) fq_dict_codes(const fq_u8 *valid, fq_u64 n, const fq_u32 *slot_of, const fq_u32 *ids, const fq_u32 *rank,
                                                     fq_u32 *codes) {
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (fq_u64)gridDim.x * blockDim.x)
    codes[i] = (valid && !valid[i]) ? 0u : rank[ids[slot_of[i]]];
}

// take, step 1: lens[i] = length of string rows[i] (0 for a NULL output slot); lens[n] = 0 so that the exclusive scan of
// n + 1 entries ends with the total; *total (u64) = the sum, to check the int32 offset limit before the offsets are used
// (total[1] != 0: some row index was out of range; such a slot is taken as empty)
__global__ void __launch_bounds__(256) fq_utf8_lens(const int *off, fq_u64 src_len, const fq_u32 *rows, const fq_u8 *rows_valid, fq_u64 n,
                                                    fq_u32 *lens, unsigned long long *total) {
  unsigned long long t = 0;
  for (fq_u64 i = (fq_u64)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += (fq_u64)gridDim.x * blockDim.x) {
    fq_u32 l = 0;
    if (i < n && (!rows_valid || rows_valid[i])) {
      if (rows[i] < src_len) l = (fq_u32)(off[rows[i] + 1] - off[rows[i]]);
      else total[1] = 1;
    }
    lens[i] = l;
    t += l;
  }
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  if ((threadIdx.x & 31) == 0 && t) atomicAdd(total, t);
}

// take, step 2: one warp per output string copies its bytes (coalesced for long strings, one round for short ones)
__global__ void __launch_bounds__(256) fq_utf8_gather_bytes(const int *off, const unsigned char *data, const fq_u32 *rows, const fq_u8 *rows_valid,
                                                            fq_u64 n, const int *out_off, unsigned char *out) {
  const fq_u64 warp = ((fq_u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, warps = ((fq_u64)gridDim.x * blockDim.x) >> 5;
  const unsigned lane = threadIdx.x & 31;
  for (fq_u64 i = warp; i < n; i += warps) {
    const fq_u32 len = (fq_u32)(out_off[i + 1] - out_off[i]);
    if (len == 0) continue;   // NULL slots and empty strings
    const unsigned char *s = data + off[rows[i]];
    unsigned char *d = out + out_off[i];
    for (fq_u32 b = lane; b < len; b += 32) d[b] = s[b];
  }
}

// (lower, upper) bound of `x` in a sorted dictionary of d strings: first index >= x, first index > x
__global__ void fq_utf8_bounds_kernel(const int *off, const unsigned char *data, fq_u64 d, const unsigned char *x, fq_u32 lx,
                                      unsigned long long *out) {
  for (int upper = 0; upper < 2; upper++) {
    fq_u64 lo = 0, hi = d;
    while (lo < hi) {
      const fq_u64 mid = (lo + hi) / 2;
      const int c = fq_utf8_cmp(data + off[mid], (fq_u32)(off[mid + 1] - off[mid]), x, lx);
      if (c < 0 || (upper && c == 0)) lo = mid + 1;
      else hi = mid;
    }
    out[upper] = lo;
  }
}
