/* octomap_msg.c -- the octomap_msgs/Octomap recipe of include/d2pc_b200.h in plain C (test infrastructure, not product
 * code): the known voxels sorted in Morton order (d2pc_occupancy_voxels' output) to the full or binary data, the way
 * csrc/occupancy.cu builds it -- each voxel's first level s and leaf level lambda, record offsets by a prefix sum, the
 * parent of a voxel's first node by a binary search, child bits ORed into parents, values maxed level by level.
 * Morton codes are the library's csrc/map_math.h. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "map_math.h"

static uint32_t ordered(uint32_t f) { return f ^ ((f >> 31) ? 0xffffffffu : 0x80000000u); }
static uint32_t unordered(uint32_t o) { return o ^ ((o >> 31) ? 0x80000000u : 0xffffffffu); }

/* keys packed kx | ky << 16 | kz << 32 in Morton order, log-odds as float bits.  Returns the data size; writes it to
 * out when cap suffices.  -1 (as size_t) when memory runs out. */
size_t d2pc_octomap_ref(const uint64_t *keys, const uint32_t *lo, size_t n, int binary, float occ_thres, uint8_t *out,
                        size_t cap) {
  if (n == 0) return 0;
  uint64_t *m = malloc(n * 8), *off = malloc((n + 1) * 8), *up = malloc(n * 8);
  uint32_t *D = malloc(n * 4);
  uint8_t *s = malloc(n), *lam = malloc(n);
  uint32_t *vmax = NULL;
  size_t total = 0;
  if (!m || !off || !up || !D || !s || !lam) {
    total = (size_t)-1;
    goto done;
  }
  for (size_t i = 0; i < n; ++i)
    m[i] = d2pc_map_morton((uint16_t)keys[i], (uint16_t)(keys[i] >> 16), (uint16_t)(keys[i] >> 32));
  for (size_t i = 0; i < n; ++i) {
    s[i] = 0;
    D[i] = i ? D[i - 1] + (lo[i] != lo[i - 1]) : 0;
    if (i) {
      int h = 63;
      while (!(((m[i] ^ m[i - 1]) >> h) & 1)) --h;
      s[i] = (uint8_t)(16 - h / 3);
    }
  }
  for (size_t i = 0; i < n; ++i) {
    lam[i] = 16;
    for (int L = 15; L >= 0; --L) {
      const uint64_t size = 1ull << (3 * (16 - L)), o = m[i] & (size - 1);
      if (size > n || o > i) break;
      const uint64_t a = i - o, b = a + size - 1;
      if (b >= n || m[a] != m[i] - o || m[b] != m[i] - o + size - 1 || D[a] != D[b]) break;
      lam[i] = (uint8_t)L;
    }
  }
  off[0] = 0;
  for (size_t i = 0; i < n; ++i) off[i + 1] = off[i] + (lam[i] < s[i] ? 0 : lam[i] - s[i] + (binary ? 0 : 1));
  total = off[n] * (binary ? 2 : 5);
  if (total > cap || !out) goto done;
  memset(out, 0, total);
  if (!binary && !(vmax = calloc(off[n], 4))) {
    total = (size_t)-1;
    goto done;
  }
  for (size_t i = 0; i < n; ++i) {
    if (lam[i] < s[i]) continue;
    if (s[i] > 0) {
      const uint32_t P = s[i] - 1u;
      const uint64_t base = m[i] & ~((1ull << (3 * (16 - P))) - 1);
      size_t a = 0, b = i - 1;
      while (a < b) {
        const size_t mid = a + (b - a) / 2;
        if (m[mid] < base) a = mid + 1;
        else b = mid;
      }
      up[i] = off[a] + P - s[a];
    }
    for (uint32_t L = s[i] > 0 ? s[i] : 1; L <= lam[i]; ++L) {
      const uint64_t parent = L == s[i] ? up[i] : off[i] + (L - 1 - s[i]);
      const uint32_t c = (uint32_t)(m[i] >> (3 * (16 - L))) & 7u;
      if (binary) {
        float v;
        memcpy(&v, &lo[i], 4);
        const uint32_t code = L < lam[i] ? 3u : (v >= occ_thres ? 2u : 1u), bits = code << (2 * c);
        out[2 * parent] |= (uint8_t)bits, out[2 * parent + 1] |= (uint8_t)(bits >> 8);
      } else {
        out[5 * parent + 4] |= (uint8_t)(1u << c);
      }
    }
  }
  if (!binary) {
    for (uint32_t L = 16; L >= 1; --L)
      for (size_t i = 0; i < n; ++i) {
        if (L < s[i] || L > lam[i]) continue;
        const uint64_t r = off[i] + (L - s[i]), parent = L == s[i] ? up[i] : r - 1;
        const uint32_t v = L == lam[i] ? ordered(lo[i]) : vmax[r];
        if (v > vmax[parent]) vmax[parent] = v;
      }
    for (size_t i = 0; i < n; ++i)
      for (uint32_t L = s[i]; L <= lam[i]; ++L) {
        const uint64_t r = off[i] + (L - s[i]);
        const uint32_t f = L == lam[i] ? lo[i] : unordered(vmax[r]);
        memcpy(out + 5 * r, &f, 4);
      }
  }
done:
  free(vmax), free(m), free(off), free(up), free(D), free(s), free(lam);
  return total;
}
