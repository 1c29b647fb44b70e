/*
 * tests/pbvi_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement of the offline PBVI solver of csrc/pbvi.cu in the product's
 * own, fully defined arithmetic (DESIGN.md section 7a): belief-set expansion
 * (expand_belief_set) and the backup (backup_on_device) with the hand-written
 * contraction, whose every R[o][b][i] is ONE ascending FMA chain from +0.
 * Everything else follows the reference's order, so the product's alpha
 * vectors, actions and belief sets can be compared with this file bit for bit
 * on any input -- not only where no arg-max is decided by the last bits.
 *
 * Built from oracle/pomdp_oracle.c (included unchanged: model tables, Bayes
 * update, normalisation, glibc rand()).  Device arithmetic of the product is
 * reproduced as there: FTZ+DAZ set in MXCSR and fmaf() where the kernel uses
 * fma.rn.ftz (Gamma_ao); fmaf() with subnormals kept where it uses
 * __fmaf_rn (the contraction); separately rounded mul / add elsewhere.
 * MXCSR is per thread, so every OpenMP region sets the mode it needs in each
 * thread and restores it.  Compiled by tests/pbvi_oracle_py.py with
 * -O2 -ffp-contract=off -fopenmp.
 *
 * The contraction is kept DENSE on purpose (all cells, never the live-cell
 * list of the kernel): equality with the product then also shows that the
 * kernel's skipping of dead cells leaves every chain unchanged.
 */
#include "../oracle/pomdp_oracle.c"

#if defined(__x86_64__)
#define FP_MODE(ftz)                                                   \
  const unsigned int fp_saved_ = _mm_getcsr();                         \
  _mm_setcsr((ftz) ? (fp_saved_ | 0x8040u) : (fp_saved_ & ~0x8040u))
#define FP_RESTORE() _mm_setcsr(fp_saved_)
#else
#define FP_MODE(ftz)
#define FP_RESTORE()
#endif

/* max_backup_iterations of the reference (pbvi.cu reference_backup_iterations):
 * float arithmetic as written. */
uint32_t pbvi_oracle_reference_iterations(float gamma) {
  return (uint32_t)ceilf(logf(1.0e-3f / 5.0f) / logf(gamma));
}

/* ---------------------------------------------------------------- backup -- */
/* pbvi_gamma_ao_kernel for action a and all 16 observations, FTZ on:
 *   tm[k] = T[s][a][k] * L[n_k][o]   (in-map neighbours k)
 *   G[o][i][s] = (fma chain from +0 over in-map k ascending of alpha_i[n_k] * tm[k]) * gamma */
ORACLE_CLONES
static void gamma_ao_rows(int32_t h, int32_t w, int32_t n, float gamma, int a, int o,
                          const float* tp, const float* mp, const float* alphas, float* G) {
  const int64_t hw = (int64_t)h * w;
  for (int64_t s = 0; s < hw; ++s) {
    const int64_t x = s % w, y = s / w;
    float tm[9];
    int64_t nidx[9];
    for (int k = 0; k < 9; ++k) {
      const int64_t nx = x + k % 3 - 1, ny = y + k / 3 - 1;
      const int in = !(nx < 0 || nx >= w || ny < 0 || ny >= h);
      nidx[k] = in ? ny * w + nx : -1;
      tm[k] = in ? tp[s * 81 + a * 9 + k] * mp[nidx[k] * 16 + o] : 0.0f;
    }
    for (int32_t i = 0; i < n; ++i) {
      const float* al = alphas + (int64_t)i * hw;
      float acc = 0.0f;
      for (int k = 0; k < 9; ++k)
        if (nidx[k] >= 0) acc = fmaf(al[nidx[k]], tm[k], acc);
      G[((int64_t)o * n + i) * hw + s] = acc * gamma;
    }
  }
}

static void gamma_ao(int32_t h, int32_t w, int32_t n, float gamma, int32_t a,
                     const float* tp, const float* mp, const float* alphas, float* G) {
#pragma omp parallel
  {
    FP_MODE(1);
#pragma omp for schedule(static)
    for (int o = 0; o < 16; ++o) gamma_ao_rows(h, w, n, gamma, a, o, tp, mp, alphas, G);
    FP_RESTORE();
  }
}

/* pbvi_sgemm_tn_kernel for one (o, b), dense, FTZ off:
 *   R[b][i] = fma chain from +0 over ALL cells s ascending of G[i][s] * B[b][s].
 * Eight independent chains at a time; each chain is still one ordered chain. */
ORACLE_CLONES
static void contract_row(int32_t n, int64_t hw, const float* G, const float* Bb, float* Rb) {
  int32_t i = 0;
  for (; i + 8 <= n; i += 8) {
    float acc[8] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    const float* g = G + (int64_t)i * hw;
    for (int64_t s = 0; s < hw; ++s) {
      const float bv = Bb[s];
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(g[(int64_t)j * hw + s], bv, acc[j]);
    }
    for (int j = 0; j < 8; ++j) Rb[i + j] = acc[j];
  }
  for (; i < n; ++i) {
    const float* g = G + (int64_t)i * hw;
    float acc = 0.0f;
    for (int64_t s = 0; s < hw; ++s) acc = fmaf(g[s], Bb[s], acc);
    Rb[i] = acc;
  }
}

/* R[o][b][i] for n_o stacked contractions: G [n_o][n][hw], B [n][hw]. */
void pbvi_oracle_contract(int32_t n_o, int32_t n, int64_t hw, const float* G, const float* B,
                          float* R) {
#pragma omp parallel
  {
    FP_MODE(0);
#pragma omp for schedule(dynamic, 4)
    for (int64_t ob = 0; ob < (int64_t)n_o * n; ++ob) {
      const int64_t o = ob / n, b = ob % n;
      contract_row(n, hw, G + o * n * hw, B + b * hw, R + (o * n + b) * n);
    }
    FP_RESTORE();
  }
}

/* backupAlphaVectors in the product's order, from zero alpha vectors.
 * B [n][hw]; alphas [n][hw] and actions [n] out; argmax (optional) [9][16][n]:
 * the Gamma_ao vector each belief picked in the LAST iteration, per action and
 * observation.  iterations == 0: the reference's count.  Returns the count run. */
uint32_t pbvi_oracle_backup(int32_t h, int32_t w, float gamma, const float* tp, const float* mp,
                            const float* sr, int32_t n, const float* B, uint32_t iterations,
                            float* alphas, uint8_t* actions, int32_t* argmax) {
  const int64_t hw = (int64_t)h * w;
  if (iterations == 0) iterations = pbvi_oracle_reference_iterations(gamma);
  float* G = (float*)malloc((size_t)16 * n * hw * sizeof(float));
  float* GA = (float*)malloc((size_t)9 * n * hw * sizeof(float));
  float* R = (float*)malloc((size_t)16 * n * n * sizeof(float));
  int32_t* idx = (int32_t*)malloc((size_t)16 * n * sizeof(int32_t));
  float* rew = (float*)malloc((size_t)9 * n * sizeof(float));
  memset(alphas, 0, (size_t)n * hw * sizeof(float));
  memset(actions, 0, (size_t)n);
  for (uint32_t it = 0; it < iterations; ++it) {
    for (int a = 0; a < 9; ++a) {
      gamma_ao(h, w, n, gamma, a, tp, mp, alphas, G);
      pbvi_oracle_contract(16, n, hw, G, B, R);
      /* pbvi_argmax_kernel: first maximum over i (std::max_element) */
      for (int64_t row = 0; row < 16 * (int64_t)n; ++row) {
        const float* r = R + row * n;
        int32_t best = 0;
        for (int32_t i = 1; i < n; ++i)
          if (r[best] < r[i]) best = i;
        idx[row] = best;
      }
      if (argmax && it + 1 == iterations)
        memcpy(argmax + (int64_t)a * 16 * n, idx, (size_t)16 * n * sizeof(int32_t));
      /* pbvi_accumulate_kernel: R(:,a), then Gamma_ao[o][argmax] + acc, o ascending */
      for (int32_t b = 0; b < n; ++b)
        for (int64_t s = 0; s < hw; ++s) {
          float acc = sr[s * 9 + a];
          for (int o = 0; o < 16; ++o) acc = G[((int64_t)o * n + idx[o * n + b]) * hw + s] + acc;
          GA[((int64_t)a * n + b) * hw + s] = acc;
        }
    }
    /* pbvi_rewards_kernel: rounded multiply, then rounded add, cells ascending */
    for (int32_t b = 0; b < n; ++b)
      for (int a = 0; a < 9; ++a) {
        const float* g = GA + ((int64_t)a * n + b) * hw;
        float acc = 0.0f;
        for (int64_t s = 0; s < hw; ++s) acc = acc + B[b * hw + s] * g[s];
        rew[b * 9 + a] = acc;
      }
    /* pbvi_select_kernel: first action strictly above all earlier ones, from -FLT_MAX;
     * the new vectors are visible only from the next iteration on */
    for (int32_t b = 0; b < n; ++b) {
      float opt = -FLT_MAX;
      int oa = 0;
      for (int a = 0; a < 9; ++a)
        if (rew[b * 9 + a] > opt) { opt = rew[b * 9 + a]; oa = a; }
      memcpy(alphas + b * hw, GA + ((int64_t)oa * n + b) * hw, (size_t)hw * sizeof(float));
      actions[b] = (uint8_t)oa;
    }
  }
  free(G); free(GA); free(R); free(idx); free(rew);
  return iterations;
}

/* ------------------------------------------------------------- expansion -- */
/* libstdc++'s __adjust_heap / __push_heap / make_heap / sort_heap on size_t
 * indices with comp(i, j) = key[i] > key[j]: what the reference's
 * partial_sort(begin, END, begin + 100) amounts to (a full heap sort).
 * Transcribed so that ties fall the same way. */
static int farther(const float* key, size_t i, size_t j) { return key[i] > key[j]; }

static void push_heap_(size_t* first, int64_t hole, int64_t top, size_t value, const float* key) {
  int64_t parent = (hole - 1) / 2;
  while (hole > top && farther(key, first[parent], value)) {
    first[hole] = first[parent];
    hole = parent;
    parent = (hole - 1) / 2;
  }
  first[hole] = value;
}

static void adjust_heap_(size_t* first, int64_t hole, int64_t len, size_t value,
                         const float* key) {
  const int64_t top = hole;
  int64_t second = hole;
  while (second < (len - 1) / 2) {
    second = 2 * (second + 1);
    if (farther(key, first[second], first[second - 1])) second--;
    first[hole] = first[second];
    hole = second;
  }
  if ((len & 1) == 0 && second == (len - 2) / 2) {
    second = 2 * (second + 1);
    first[hole] = first[second - 1];
    hole = second - 1;
  }
  push_heap_(first, hole, top, value, key);
}

static void heap_sort_farthest_first(size_t* first, int64_t len, const float* key) {
  if (len < 2) return;
  for (int64_t parent = (len - 2) / 2;; --parent) {       /* make_heap */
    adjust_heap_(first, parent, len, first[parent], key);
    if (parent == 0) break;
  }
  for (int64_t last = len - 1; last > 0; --last) {        /* sort_heap: pop_heap */
    const size_t value = first[last];
    first[last] = first[0];
    adjust_heap_(first, 0, last, value, key);
  }
}

/* generateBeliefSet as expand_belief_set runs it.  b0 [hw]; out [max_size][hw]. */
void pbvi_oracle_expand(int32_t h, int32_t w, const float* tp, const float* mp, const float* b0,
                        uint32_t max_size, uint32_t rand_seed, float* out) {
  const int64_t hw = (int64_t)h * w;
  glibc_rand_t rng;
  oracle_glibc_srand(&rng, rand_seed ? rand_seed : 1);
  memcpy(out, b0, (size_t)hw * sizeof(float));
  uint32_t size = 1;
  while (size < max_size) {
    const int64_t n = size, nc = n * 9;
    float* draws = (float*)malloc((size_t)nc * 3 * sizeof(float));
    for (int64_t t = 0; t < nc * 3; ++t)
      draws[t] = (float)oracle_glibc_rand(&rng) / ((float)2147483647 + 1.0f);
    float* cand = (float*)malloc((size_t)nc * hw * sizeof(float));
    float* l1 = (float*)malloc((size_t)nc * sizeof(float));
#pragma omp parallel
    {
      FP_MODE(0);
      float* prefix = (float*)malloc((size_t)hw * sizeof(float));
#pragma omp for schedule(dynamic, 1)
      for (int64_t i = 0; i < n; ++i) {
        const float* bi = out + i * hw;
        float acc = 0.0f;                                  /* partial_sum */
        for (int64_t s = 0; s < hw; ++s) { acc = acc + bi[s]; prefix[s] = acc; }
        for (int a = 0; a < 9; ++a) {
          const int64_t t = i * 9 + a;
          const float r1 = draws[3 * t], r2 = draws[3 * t + 1], r3 = draws[3 * t + 2];
          /* pbvi_sample_kernel: lower-bound search, clamped to the last cell */
          int64_t lo = 0, hi = hw;
          while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (prefix[mid] >= r1) hi = mid; else lo = mid + 1;
          }
          const int64_t s = lo < hw ? lo : hw - 1;
          float cum = 0.0f;
          int ns_local = 8, found = 0;
          for (int j = 0; j < 9; ++j) {
            const float p = tp[s * 81 + a * 9 + j];
            cum = j == 0 ? p : cum + p;
            if (!found && cum >= r2) { ns_local = j; found = 1; }
          }
          int64_t ns = (s / w + ns_local / 3 - 1) * w + (s % w + ns_local % 3 - 1);
          if (ns < 0) ns = 0;
          if (ns >= hw) ns = hw - 1;
          int z = 15;
          found = 0;
          cum = 0.0f;
          for (int j = 0; j < 16; ++j) {
            const float p = mp[ns * 16 + j];
            cum = j == 0 ? p : cum + p;
            if (!found && cum >= r3) { z = j; found = 1; }
          }
          float* c = cand + t * hw;
          oracle_pomdp_bayes_update((uint32_t)h, (uint32_t)w, tp, mp, bi, (uint8_t)a, (uint8_t)z, c);
          oracle_pomdp_normalize((uint64_t)hw, c);
        }
      }
      /* pbvi_l1_kernel: min over the set of sub, abs, add chains; a NaN sum
       * never becomes the minimum (start: FLT_MAX) */
#pragma omp for schedule(dynamic, 1)
      for (int64_t t = 0; t < nc; ++t) {
        const float* c = cand + t * hw;
        float best = FLT_MAX;
        int64_t j = 0;
        for (; j + 4 <= n; j += 4) {
          float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
          for (int64_t s = 0; s < hw; ++s)
            for (int q = 0; q < 4; ++q) acc[q] = acc[q] + fabsf(c[s] - out[(j + q) * hw + s]);
          for (int q = 0; q < 4; ++q)
            if (acc[q] < best) best = acc[q];
        }
        for (; j < n; ++j) {
          float acc = 0.0f;
          for (int64_t s = 0; s < hw; ++s) acc = acc + fabsf(c[s] - out[j * hw + s]);
          if (acc < best) best = acc;
        }
        l1[t] = best;
      }
      free(prefix);
      FP_RESTORE();
    }
    /* per belief the action whose candidate is farthest (max_element) */
    int64_t* new_bs = (int64_t*)malloc((size_t)n * sizeof(int64_t));
    float* new_bs_l1 = (float*)malloc((size_t)n * sizeof(float));
    for (int64_t i = 0; i < n; ++i) {
      const float* r = l1 + i * 9;
      int best = 0;
      for (int a = 1; a < 9; ++a)
        if (r[best] < r[a]) best = a;
      new_bs[i] = i * 9 + best;
      new_bs_l1[i] = r[best];
    }
    size_t* order = (size_t*)malloc((size_t)n * sizeof(size_t));
    for (int64_t i = 0; i < n; ++i) order[i] = (size_t)i;
    int64_t n_take = n;
    if (n >= 100) {
      heap_sort_farthest_first(order, n, new_bs_l1);
      n_take = 100;
    }
    for (int64_t k = 0; k < n_take; ++k) {
      memcpy(out + (int64_t)size * hw, cand + new_bs[order[k]] * hw, (size_t)hw * sizeof(float));
      if (++size >= max_size) break;
    }
    free(order); free(new_bs); free(new_bs_l1);
    free(draws); free(cand); free(l1);
  }
}
