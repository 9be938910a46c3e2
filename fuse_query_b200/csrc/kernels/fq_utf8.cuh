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
// fq_utf8_like_kernel matches a LIKE pattern against every string of an array (over a dictionary: once per distinct string)
// and writes one bit per row, which pipes read through an FQ_EXPR_LOOKUP node.
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

// SQL LIKE, bytewise and case-sensitive: `%` = any run of characters (newlines included), `_` = one UTF-8 code point,
// `\` makes the next pattern byte literal (the caller refuses a pattern that ends in an unpaired `\`).  Greedy matching that
// keeps one backtrack point, the last `%` seen: when the text after it fails, that `%` swallows one more code point and the
// rest of the pattern is tried again.  No recursion, O(len * plen) steps at worst.  Plain code, no intrinsics: the tests
// compile this very function for the host.
__device__ __forceinline__ bool fq_like_match(const unsigned char *s, fq_u32 len, const unsigned char *p, fq_u32 plen) {
  fq_u32 i = 0, j = 0;
  fq_u32 star_j = 0xFFFFFFFFu, star_i = 0;   // pattern position after the last `%`, text position it was resumed from
  while (i < len) {
    if (j < plen) {
      const unsigned char c = p[j];
      if (c == '%') {
        star_j = ++j;
        star_i = i;
        continue;
      }
      if (c == '_') {   // one code point: the lead byte and its continuation bytes
        i++;
        while (i < len && (s[i] & 0xC0) == 0x80) i++;
        j++;
        continue;
      }
      const bool esc = c == '\\' && j + 1 < plen;
      if (s[i] == (esc ? p[j + 1] : c)) {
        i++;
        j += esc ? 2 : 1;
        continue;
      }
    }
    if (star_j == 0xFFFFFFFFu) return false;
    star_i++;   // the last `%` takes one more code point
    while (star_i < len && (s[star_i] & 0xC0) == 0x80) star_i++;
    i = star_i;
    j = star_j;
  }
  while (j < plen && p[j] == '%') j++;
  return j == plen;
}

// bit i of `bits` (LSB-first) = string i LIKE the pattern, xor `negate`; NULL rows and the padding of the last byte get 0.
// One thread per string, one 32-bit word per warp from a ballot: no atomics.  The word is stored byte by byte where the
// column is not 4-byte aligned or ends inside it (the column holds ceil(n / 8) bytes).
__global__ void __launch_bounds__(256) fq_utf8_like_kernel(const int *off, const unsigned char *data, const fq_u8 *valid, fq_u64 n,
                                                           const unsigned char *pat, fq_u32 plen, int negate, fq_u8 *bits) {
  const unsigned lane = threadIdx.x & 31;
  const fq_u64 n_words = (n + 31) / 32, n_bytes = (n + 7) / 8;
  const bool aligned = ((unsigned long long)bits & 3) == 0;
  for (fq_u64 w = ((fq_u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_words; w += ((fq_u64)gridDim.x * blockDim.x) >> 5) {
    const fq_u64 i = w * 32 + lane;
    bool hit = false;
    if (i < n && (!valid || valid[i])) hit = fq_like_match(data + off[i], (fq_u32)(off[i + 1] - off[i]), pat, plen) != (negate != 0);
    const fq_u32 word = __ballot_sync(0xffffffffu, hit);
    if (lane == 0) {
      if (aligned && 4 * w + 4 <= n_bytes) {
        reinterpret_cast<fq_u32 *>(bits)[w] = word;
      } else {
        for (fq_u64 b = 4 * w; b < 4 * w + 4 && b < n_bytes; b++) bits[b] = (fq_u8)(word >> (8 * (b - 4 * w)));
      }
    }
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
