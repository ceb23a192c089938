// lns_chain.cuh -- body of one search chain (one warp), included INSIDE the kernels k_lns and k_lns_global (lns.cu).
//
// It is an included body rather than a device function because that is what leaves k_lns's code as it was: moved into a
// __forceinline__ function the same statements compile to other registers (k = 3, 8 chains per block: 116 -> 113) and
// the bench ran 8 % slower on a B200.  The including kernel defines, before the #include:
//   St (LnsShared | LnsGlobal) and pod_t, idx_t, dix_t, NT = 2^KK, kNone from it; a (LnsArgs), N, F, fn, smax, lane,
//   chain, b; dT[N][N] (transposed delays), w[F][N], r[F][N], K[N], slots[N] of the chain's instance; wp (the chain's
//   state, lns_chain_bytes<St>); noise0 (start temperature), u, a_d (objective weights).
// Everything here is the same code for both state placements: same random streams, evaluation and summation orders and
// decisions, so on any input both kernels take the same records bit for bit.
  // ---- per-chain state -----------------------------------------------------------------------------------
  double* lam = (double*)wp; wp += (size_t)N * 8;
  unsigned long long* loadfx = (unsigned long long*)wp; wp += (size_t)N * 8;
  float* bestv = (float*)wp; wp += ((size_t)fn * 4 + 15) & ~(size_t)15;
  unsigned char* scratch = wp; wp += lns_scratch_bytes<St>(N, F, KK, smax, a.maxslots);
  double* costT = (double*)scratch;                       // [F][NT]
  double* dp = costT + (size_t)F * NT;                    // [smax]
  float* th = (float*)scratch;                            // aliases the DP arrays (never live together)
  idx_t* thl = (idx_t*)(scratch + (size_t)(a.maxslots < F ? a.maxslots : F) * N * 4);   // sources whose threshold needs a pod scan
  idx_t* exl = (idx_t*)scratch;         // exception list, ditto
  int* npods = (int*)wp; wp += (size_t)F * 4;
  int* misc = (int*)wp; wp += 33 * 4;
  int* fl = (int*)wp; wp += (size_t)F * 4;
  pod_t* asg; uint8_t* c; pod_t* podlist;
  if constexpr (St::kGlobal) {                            // c padded: podlist stays aligned
    asg = (pod_t*)wp; wp += (size_t)fn * sizeof(pod_t);
    c = wp; wp += ((size_t)fn + 1) & ~(size_t)1;
    podlist = (pod_t*)wp; wp += (size_t)fn * sizeof(pod_t);
  } else {
    asg = (pod_t*)wp; wp += fn;
    c = wp; wp += fn;
    podlist = (pod_t*)wp; wp += fn;
  }
  uint8_t* choice = wp; wp += (size_t)F * smax;
  uint8_t* suppT = wp; wp += smax;
  uint8_t* oldT = wp; wp += F;
  uint8_t* newT = wp;
  int* Jn = misc; int* rad = misc + 4; int* mul = misc + 8; int* incT = misc + 12;      // incT[16]

  uint64_t rs = a.rng ^ (0x9E3779B97F4A7C15ull * (uint64_t)(chain + 1)) ^ (0xD1B54A32D192ED03ull * (uint64_t)(b + 1));
  lns_next(rs); lns_next(rs);

  // ---- start placement -----------------------------------------------------------------------------------
  for (int q = lane; q < fn; q += 32) c[q] = 0;
  for (int j = lane; j < N; j += 32) lam[j] = a.lam0 ? fmax(a.lam0[(int64_t)b * N + j], 0.0) : 0.0;
  __syncwarp();
  const bool from_seed = a.seeds && (!a.guide || chain < a.S);
  if (from_seed) {
    const uint8_t* seed = a.seeds + ((int64_t)b * a.S + (chain % a.S)) * fn;
    for (int q = lane; q < fn; q += 32) c[q] = seed[q] ? 1 : 0;
    __syncwarp();
    // seeds may exceed the slot count of a node (never for EFTTC output): drop the highest-numbered extras
    for (int j = lane; j < N; j += 32) { int cnt = 0; for (int f = 0; f < F; ++f) { if (c[f * N + j]) { if (cnt >= slots[j]) c[f * N + j] = 0; else ++cnt; } } }
  } else {
    // randomised rounding: per node the `slots` functions with the largest perturbed c-bar (or random without guide)
    const double amp = a.guide ? 0.02 + 0.12 * (double)((chain / 2) % 4) : 1.0;
    const double* g = a.guide ? a.guide + (int64_t)b * fn : nullptr;
    for (int j = lane; j < N; j += 32) {
      for (int cnt = 0; cnt < slots[j]; ++cnt) {
        int bf = -1; double bg = -INFINITY;
        for (int f = 0; f < F; ++f) {
          if (c[f * N + j]) continue;
          const double v = (g ? g[f * N + j] : 0.0) + amp * lns_u01(lns_mix(rs ^ ((uint64_t)(f * N + j) << 20)));
          if (v > bg) { bg = v; bf = f; }
        }
        if (bf < 0) break;
        c[bf * N + j] = 1;
      }
    }
  }
  __syncwarp();
  // every function needs a pod: put a missing one on the node where it has the most workload and a free slot,
  // else replace the pod of the function with the most pods there (lane 0; rare)
  if (lane == 0) {
    for (int f = 0; f < F; ++f) {
      int any = 0; for (int j = 0; j < N; ++j) any |= c[f * N + j];
      if (any) continue;
      int bj = -1; double bw = -1.0;
      for (int j = 0; j < N; ++j) { if (slots[j] <= 0) continue; if (w[f * N + j] > bw) { bw = w[f * N + j]; bj = j; } }
      if (bj < 0) continue;
      int cnt = 0; for (int f2 = 0; f2 < F; ++f2) cnt += c[f2 * N + bj];
      if (cnt >= slots[bj]) {
        int vf = -1, vp = 1;
        for (int f2 = 0; f2 < F; ++f2) { if (!c[f2 * N + bj]) continue; int p2 = 0; for (int j = 0; j < N; ++j) p2 += c[f2 * N + j]; if (p2 > vp) { vp = p2; vf = f2; } }
        if (vf < 0) continue;
        c[vf * N + bj] = 0;
      }
      c[f * N + bj] = 1;
    }
  }
  __syncwarp();

  // pod list of one function, ascending (ballot compaction; warp-uniform call)
  auto rebuild_pods = [&](int f) {
    int n = 0;
    for (int jb = 0; jb < N; jb += 32) {
      const int j = jb + lane;
      const bool on = j < N && c[f * N + j];
      const unsigned bal = __ballot_sync(0xffffffffu, on);
      if (on) podlist[f * N + n + __popc(bal & ((1u << lane) - 1u))] = (pod_t)j;
      n += __popc(bal);
    }
    if (lane == 0) npods[f] = n;
    __syncwarp();
  };
  // nearest priced pod of every source of f (lanes over sources, pods in a warp-uniform loop); `skip` < 0: none excluded
  auto scan_function = [&](int f) {
    const int np = npods[f];
    const pod_t* pl = podlist + f * N;
    const double* rf = r + f * N;
    for (int ib = 0; ib < N; ib += 32) {
      const int i = ib + lane;
      double best = kLnsBig; int bj = kNone;
      if (i < N) {
#pragma unroll 2
        for (int q = 0; q < np; ++q) {
          const int j = pl[q];
          const double v = dT[(dix_t)j * N + i] + lam[j] * rf[j];
          if (v < best) { best = v; bj = j; }
        }
        bestv[f * N + i] = (float)best; asg[f * N + i] = (pod_t)bj;
      }
    }
  };
  for (int f = 0; f < F; ++f) rebuild_pods(f);
  for (int f = 0; f < F; ++f) scan_function(f);
  __syncwarp();

  uint64_t dirtyF = ~0ull;             // functions whose routing changed since the node prices were last settled
  double bestu = INFINITY, bestg = -INFINITY; int best_round = -1;
  double bestg2 = INFINITY, bestu2 = INFINITY; int best_round2 = -1;
  // records of an instance: [0, chains) by the whole-flow (upper-bound) objective, [chains, 2 chains) by the priced one
  uint8_t* outc = a.out_c + ((int64_t)b * 2 * a.chains + chain) * fn;
  uint8_t* outc2 = a.out_c + ((int64_t)b * 2 * a.chains + a.chains + chain) * fn;
  // k_lns_global also returns the routing each record was taken with (asg: every source's pod)
  uint16_t* outa = St::kGlobal ? a.out_asg + ((int64_t)b * 2 * a.chains + chain) * fn : nullptr;
  uint16_t* outa2 = St::kGlobal ? a.out_asg + ((int64_t)b * 2 * a.chains + a.chains + chain) * fn : nullptr;
  const int anneal_rounds = a.rounds - a.rounds / 8;

  #pragma unroll 1
  for (int round = 0; round <= a.rounds; ++round) {
    // ---- neighbourhood: a random node and k-1 nodes near it (tournaments on d), or k random nodes ----------
    int kk = KK;
    uint64_t jm0 = 0, jm1 = 0;                       // the k nodes as a bitmask (N <= 128) ...
    int Jk[KK];                                      // ... or as a list (N > 128)
    {
      int J[KK];
      const uint64_t h0 = lns_next(rs);
      J[0] = (int)(((h0 & 0xffffffffull) * (uint64_t)N) >> 32);
      const bool local = ((h0 >> 40) & 3) != 0;
      int have = 1;
      #pragma unroll 1
      for (int tries = 0; have < KK && tries < 16 * KK; ++tries) {
        int bj = -1; double bd = INFINITY;
        const uint64_t h = lns_next(rs);
        const int tsize = local ? 1 + (int)((h >> 50) & 3) : 1;
        uint64_t hh = h;
        #pragma unroll 1
        for (int t = 0; t < tsize; ++t) {
          hh = lns_mix(hh + t);
          const int j = (int)(((hh & 0xffffffffull) * (uint64_t)N) >> 32);
          bool dup = false;
#pragma unroll
          for (int q = 0; q < KK; ++q) dup = dup || (q < have && J[q] == j);
          if (dup) continue;
          const int pick = (int)((((hh >> 32) & 0xffffull) * (uint64_t)have) >> 16);
          int jp = J[0];
#pragma unroll
          for (int q = 1; q < KK; ++q) if (q == pick) jp = J[q];
          const double dv = dT[(dix_t)j * N + jp];
          if (dv < bd) { bd = dv; bj = j; }
        }
        if (bj >= 0) {
#pragma unroll
          for (int q = 1; q < KK; ++q) if (q == have) J[q] = bj;
          ++have;
        }
      }
      kk = have;
      // state space of the slot counters must fit: drop trailing nodes otherwise
      int S_ = 1, fit = 0;
#pragma unroll
      for (int q = 0; q < KK; ++q) {
        if (q < kk && fit == q) { const int rd = slots[J[q]] + 1; if ((int64_t)S_ * rd <= smax) { S_ *= rd; ++fit; } }
      }
      kk = fit;
      if (lane == 0) {
        int mu_ = 1;
#pragma unroll
        for (int q = 0; q < KK; ++q) if (q < kk) { Jn[q] = J[q]; rad[q] = slots[J[q]] + 1; mul[q] = mu_; mu_ *= rad[q]; }
        misc[32] = mu_;                                    // number of states
      }
#pragma unroll
      for (int q = 0; q < KK; ++q) {
        if constexpr (St::kGlobal) Jk[q] = q < kk ? J[q] : -1;
        else if (q < kk) { if (J[q] < 64) jm0 |= 1ull << J[q]; else jm1 |= 1ull << (J[q] - 64); }
      }
    }
    __syncwarp();
    auto inJ = [&](int j) -> bool {
      if constexpr (St::kGlobal) {
        bool in = false;
#pragma unroll
        for (int q = 0; q < KK; ++q) in = in || Jk[q] == j;
        return in;
      } else {
        return j < 64 ? (jm0 >> j) & 1 : (j < 128 ? (jm1 >> (j - 64)) & 1 : false);
      }
    };

    // ---- CPU loads at the current prices; dual ascent on the prices of overloaded / priced nodes -----------------
    // A node is (re)priced when it is overloaded or carries a price.  Price of node jj = the threshold at which enough of its flows leave:  a source (f,i) uses jj
    // while  lam_jj < th = (best priced alternative - d[i,jj]) / r[f,jj];  flows leave in ascending th until the
    // rest fits K_jj; ties with the alternative (th = 0) leave first, at a price of 1e-9.
    bool overloaded = false, settled = false;
    double ucost = 0.0;
    // the state of a node depends only on the functions with a pod on it: a price is re-derived when the node is
    // overloaded, or when one of its functions changed pods (last apply) or was re-routed by another node's new price
    uint64_t dirty_now = dirtyF;
    const int max_pass = N <= 32 ? 12 : 4;              // small instances with most CPU rows binding need more sweeps of the ascent
    #pragma unroll 1
    for (int pass = 0; pass < max_pass; ++pass) {
      #pragma unroll 1
      for (int j = lane; j < N; j += 32) loadfx[j] = 0ull;
      __syncwarp();
      double up = 0.0;
      #pragma unroll 1
      for (int fi = lane; fi < fn; fi += 32) {
        const int bj = asg[fi];
        if (bj == kNone) continue;
        const int f = fi / N, i = fi - f * N;
        const double wv = w[fi];
        const double ld = wv * r[f * N + bj];
        if (ld > 0.0) atomicAdd(&loadfx[bj], (unsigned long long)(fmin(ld, 1e9) * kFxScale + 0.5));
        if (wv > 0.0) up += wv * dT[(dix_t)bj * N + i];
      }
      ucost = warp_sum(up);                              // delay of the whole-flow routing at the current prices
      __syncwarp();
      bool changed = false; overloaded = false;
      #pragma unroll 1
      for (int jb = 0; jb < N; jb += 32) {
        const int j = jb + lane;
        bool need = false, over = false;
        if (j < N) {
          const double ld = (double)loadfx[j] * (1.0 / kFxScale);
          over = ld > K[j] + 1e-7;
          uint64_t on = 0;
          if (F <= 64) { for (int f = 0; f < F; ++f) if (c[f * N + j]) on |= 1ull << f; } else on = ~0ull;
          need = over || (lam[j] > 0.0 && (on & dirty_now) != 0);
        }
        unsigned todo = __ballot_sync(0xffffffffu, need);
        overloaded = overloaded || __any_sync(0xffffffffu, over);
        if (pass == max_pass - 1) continue;                // last pass only evaluates
        #pragma unroll 1
        while (todo) {
          const int jj = jb + (__ffs(todo) - 1); todo &= todo - 1;
          int nf = 0;
          #pragma unroll 1
          for (int fb = 0; fb < F; fb += 32) {
            const int f = fb + lane;
            const bool on = f < F && c[f * N + jj];
            const unsigned bal = __ballot_sync(0xffffffffu, on);
            if (on) fl[nf + __popc(bal & ((1u << lane) - 1u))] = f;
            nf += __popc(bal);
          }
          __syncwarp();
          const int M = nf * N;
          // thresholds: a source whose nearest priced pod is not jj has that pod as its alternative; the sources
          // currently ON jj need their second-best pod -- a pod scan, done for the compacted list of them only
          double tot = 0.0; int nscan = 0;
          #pragma unroll 1
          for (int tb = 0; tb < M; tb += 32) {
            const int t = tb + lane;
            bool scan = false;
            if (t < M) {
              const int z = t / N, i = t - z * N, f = fl[z];
              const double rfj = r[f * N + jj], av = w[f * N + i] * rfj;
              float tv = -1.0f;                              // never uses jj
              if (av > 0.0) {
                if (asg[f * N + i] != jj) {
                  const double tq = ((double)bestv[f * N + i] - dT[(dix_t)jj * N + i]) / rfj;
                  if (tq >= 0.0) { tv = bestv[f * N + i] >= 0.5f * (float)kLnsBig ? INFINITY : (float)fmin(tq, 1e30); tot += av; }
                } else scan = true;
              }
              th[t] = tv;
            }
            const unsigned bal = __ballot_sync(0xffffffffu, scan);
            if (scan) thl[nscan + __popc(bal & ((1u << lane) - 1u))] = (idx_t)t;
            nscan += __popc(bal);
          }
          __syncwarp();
          #pragma unroll 1
          for (int e = lane; e < nscan; e += 32) {
            const int t = thl[e], z = t / N, i = t - z * N, f = fl[z];
            const double* rf = r + f * N; const pod_t* pl = podlist + f * N; const int np = npods[f];
            const double rfj = rf[jj];
            double alt = kLnsBig;
            #pragma unroll 1
            for (int q = 0; q < np; ++q) { const int j2 = pl[q]; if (j2 == jj) continue; const double v = dT[(dix_t)j2 * N + i] + lam[j2] * rf[j2]; if (v < alt) alt = v; }
            const double tq = (alt - dT[(dix_t)jj * N + i]) / rfj;
            if (tq >= 0.0) { th[t] = alt >= 0.5 * kLnsBig ? INFINITY : (float)fmin(tq, 1e30); tot += w[f * N + i] * rfj; }   // no other pod: cannot leave
          }
          tot = warp_sum(tot);
          __syncwarp();
          double nl = 0.0;
          if (tot > K[jj] + 1e-9) {
            float last = -1.0f;
            #pragma unroll 1
            for (int it = 0; it < M && tot > K[jj] + 1e-9; ++it) {
              unsigned mn = 0xffffffffu;
              #pragma unroll 1
              for (int t = lane; t < M; t += 32) { const float tv = th[t]; if (tv > last) mn = min(mn, __float_as_uint(tv)); }
              mn = __reduce_min_sync(0xffffffffu, mn);
              if (mn >= 0x7f800000u) break;                 // nothing movable left: the node stays overloaded (never recorded)
              last = __uint_as_float(mn);
              double rem = 0.0;
              #pragma unroll 1
              for (int t = lane; t < M; t += 32) if (th[t] == last) { const int z = t / N; rem += w[fl[z] * N + (t - z * N)] * r[fl[z] * N + jj]; }
              tot -= warp_sum(rem);
            }
            nl = (double)fmaxf(last, 0.0f) * (1.0 + 2e-6) + 1e-9;
          }
          const bool ch = fabs(nl - lam[jj]) > 1e-10 * (1.0 + nl);
          __syncwarp();
          if (ch) {
            changed = true;
            if (lane == 0) lam[jj] = nl;
            __syncwarp();
            #pragma unroll 1
            for (int z = 0; z < nf; ++z) { scan_function(fl[z]); dirty_now |= F <= 64 ? 1ull << fl[z] : ~0ull; }   // their sources see a new price on jj
            __syncwarp();
          }
        }
      }
      if (!changed) { settled = true; break; }
    }
    dirtyF = settled ? 0ull : dirty_now;
    // ---- record ---------------------------------------------------------------------------------------------------
    // With no node overloaded, routing every source WHOLE to its nearest priced pod is a feasible point of the MIP
    // (pods that end up unused are closed, the others serve at least one whole source: C1b holds), so its delay
    // `ucost` is an upper bound of the placement's true objective and the priced cost g a lower bound; they differ
    // by sum_j lam_j (K_j - load_j).  Chains record by the upper bound: it can only be improved by the exact routing
    // LP afterwards (split flows), never be a mirage of loose prices.
    {
      double gp = 0.0;
      #pragma unroll 1
      for (int fi = lane; fi < fn; fi += 32) { const double wv = w[fi]; if (wv > 0.0) gp += wv * (double)bestv[fi]; }
      #pragma unroll 1
      for (int j = lane; j < N; j += 32) gp -= lam[j] * K[j];
      double g = warp_sum(gp), uval = ucost;
      if (u != 0.0) {
        int act = 0;
        #pragma unroll 1
        for (int j = lane; j < N; j += 32) { int any = 0; for (int f = 0; f < F; ++f) any |= c[f * N + j]; act += any; }
        act = __reduce_add_sync(0xffffffffu, act);
        g += u * (double)act; uval += u * (double)act;
      }
      bool unserved = false;
      #pragma unroll 1
      for (int fi = lane; fi < fn; fi += 32) unserved = unserved || asg[fi] == kNone;
      unserved = __any_sync(0xffffffffu, unserved);
      if (!overloaded && !unserved && uval < bestu - 1e-9 * (1.0 + fabs(uval))) {
        bestu = uval; bestg = g; best_round = round;
        #pragma unroll 1
        for (int q = lane; q < fn; q += 32) outc[q] = c[q];
        if constexpr (St::kGlobal) for (int q = lane; q < fn; q += 32) outa[q] = asg[q];
      }
      // second record, by the lower bound: where the optimal routing splits flows, g is the LP value and the whole-flow
      // value overstates it by sum_j lam_j (K_j - load_j) -- 15 % on a 20-node instance whose optimum splits a heavy flow.
      // Only with settled prices; both records are priced exactly by the caller.
      if (!overloaded && !unserved && settled && g < bestg2 - 1e-9 * (1.0 + fabs(g))) {
        bestg2 = g; bestu2 = uval; best_round2 = round;
        #pragma unroll 1
        for (int q = lane; q < fn; q += 32) outc2[q] = c[q];
        if constexpr (St::kGlobal) for (int q = lane; q < fn; q += 32) outa2[q] = asg[q];
      }
    }
    if (round == a.rounds) break;
    if (kk == 0) continue;

    // ---- sources served from the k nodes: their nearest pod OUTSIDE the k nodes (compacted list, then a scan) ------
    int nex = 0;
    #pragma unroll 1
    for (int fb = 0; fb < fn; fb += 32) {
      const int fi = fb + lane;
      const bool ex = fi < fn && asg[fi] != kNone && inJ(asg[fi]);
      const unsigned bal = __ballot_sync(0xffffffffu, ex);
      if (ex) exl[nex + __popc(bal & ((1u << lane) - 1u))] = (idx_t)fi;
      nex += __popc(bal);
    }
    __syncwarp();
    #pragma unroll 1
    for (int e = lane; e < nex; e += 32) {
      const int fi = exl[e], f = fi / N, i = fi - f * N;
      const pod_t* pl = podlist + f * N; const double* rf = r + f * N; const int np = npods[f];
      double best = kLnsBig; int bj = kNone;
      #pragma unroll 1
      for (int q = 0; q < np; ++q) {
        const int j = pl[q];
        if (inJ(j)) continue;
        const double v = dT[(dix_t)j * N + i] + lam[j] * rf[j];
        if (v < best) { best = v; bj = j; }
      }
      bestv[fi] = (float)best; asg[fi] = (pod_t)bj;      // (bestv, asg) now describe "the k nodes closed" for every source
    }
    __syncwarp();

    // ---- cost of every subset T of the k nodes, per function (lanes over sources, NT accumulators per lane) ------
    const double temp = round < anneal_rounds ? noise0 * (1.0 - (double)round / (double)anneal_rounds) : 0.0;
    const uint64_t rround = lns_next(rs);
    const int Tvalid = (1 << kk) - 1;
    int Jr[KK];
#pragma unroll
    for (int q = 0; q < KK; ++q) Jr[q] = q < kk ? Jn[q] : 0;
    #pragma unroll 1
    for (int f = lane; f < F; f += 32) {
      int ot = 0;
#pragma unroll
      for (int q = 0; q < KK; ++q) if (q < kk && c[f * N + Jr[q]]) ot |= 1 << q;
      oldT[f] = (uint8_t)ot;
    }
    __syncwarp();
    #pragma unroll 1
    for (int f = 0; f < F; ++f) {
      double pj[KK];
#pragma unroll
      for (int q = 0; q < KK; ++q) pj[q] = q < kk ? lam[Jr[q]] * r[f * N + Jr[q]] : kLnsBig;
      double acc[NT];
#pragma unroll
      for (int t = 0; t < NT; ++t) acc[t] = 0.0;
      #pragma unroll 1
      for (int ib = 0; ib < N; ib += 32) {
        const int i = ib + lane;
        if (i >= N) continue;
        const double wv = w[f * N + i];
        if (wv == 0.0) continue;
        double val[NT];
        val[0] = (double)bestv[f * N + i];
        double vq[KK];
#pragma unroll
        for (int q = 0; q < KK; ++q) vq[q] = dT[(dix_t)Jr[q] * N + i] + pj[q];
#pragma unroll
        for (int t = 1; t < NT; ++t) val[t] = fmin(val[t & (t - 1)], vq[__ffs(t) - 1]);
#pragma unroll
        for (int t = 0; t < NT; ++t) acc[t] += wv * val[t];
      }
      const double tot = lns_multi_reduce<NT>(acc, lane);
      const int T = lane >> (5 - KK);
      if ((lane & ((32 >> KK) - 1)) == 0) {
        double v = tot;
        if (temp > 0.0) v += temp * lns_u01(lns_mix(rround ^ ((uint64_t)(f * 64 + T) << 8))) * (double)__popc(T);
        const bool outside = npods[f] - __popc((unsigned)oldT[f]) > 0;
        if ((T & ~Tvalid) != 0 || (T == 0 && !outside)) v = INFINITY;     // dropped node / the function would lose its last pod
        costT[f * NT + T] = v;
      }
    }
    __syncwarp();

    // ---- DP over functions, state = slot counters of the k nodes -----------------------------------------------
    const int S_ = misc[32];
    #pragma unroll 1
    for (int T = lane; T < NT; T += 32) { int s = 0; for (int q = 0; q < kk; ++q) if ((T >> q) & 1) s += mul[q]; incT[T] = s; }
    #pragma unroll 1
    for (int s = lane; s < S_; s += 32) {
      int supp = 0;
      #pragma unroll 1
      for (int q = 0; q < kk; ++q) if ((s / mul[q]) % rad[q] > 0) supp |= 1 << q;
      suppT[s] = (uint8_t)supp;
      dp[s] = s == 0 ? 0.0 : INFINITY;
    }
    __syncwarp();
    // one array, updated in place: state s2 reads only states s2 - inc(T) <= s2, so the states are processed in
    // descending blocks of 32 and every lane has read before any lane stores its block -- the reads see the values
    // of the previous function exactly as with two arrays
    int mulr[KK];                                       // slot increment of each node (k = 4 candidate loop)
#pragma unroll
    for (int q = 0; q < KK; ++q) mulr[q] = q < kk ? mul[q] : 0;
    #pragma unroll 1
    for (int f = 0; f < F; ++f) {
      const double* ct = costT + f * NT;
      #pragma unroll 1
      for (int sb = (S_ - 1) & ~31; sb >= 0; sb -= 32) {
        const int s2 = sb + lane;
        double best = INFINITY; int bt = 0;
        if (s2 < S_) {
          // the subsets of the used nodes in descending order (ties keep the largest T)
          const int supp = suppT[s2];
          if constexpr (KK == 4) {
            // all 16 subsets unrolled, increments in registers: the loads of one state do not depend on each other
            // (measured faster at k = 4; slower at k = 3, where a state has ~5 subsets and the build has 80 registers)
#pragma unroll
            for (int T = NT - 1; T >= 0; --T) {
              if ((T & ~supp) != 0) continue;
              int inc = 0;
#pragma unroll
              for (int q = 0; q < KK; ++q) if ((T >> q) & 1) inc += mulr[q];
              const double v = dp[s2 - inc] + ct[T];
              if (v < best) { best = v; bt = T; }
            }
          } else {
            int Ts = supp;
            #pragma unroll 1
            while (true) {
              const double v = dp[s2 - incT[Ts]] + ct[Ts];
              if (v < best) { best = v; bt = Ts; }
              if (Ts == 0) break;
              Ts = (Ts - 1) & supp;
            }
          }
        }
        __syncwarp();
        if (s2 < S_) { dp[s2] = best; choice[f * smax + s2] = (uint8_t)bt; }
      }
      __syncwarp();
    }
    // best final state (utilisation: an empty node costs nothing, a used one u)
    double bv = INFINITY; int bs = 0x7fffffff;
    #pragma unroll 1
    for (int s = lane; s < S_; s += 32) {
      double v = dp[s];
      if (u != 0.0) v += u * (double)__popc((unsigned)suppT[s]);
      if (v < bv) { bv = v; bs = s; }
    }
    #pragma unroll 1
    for (int o = 16; o > 0; o >>= 1) {
      const double v2 = __shfl_xor_sync(0xffffffffu, bv, o); const int s2 = __shfl_xor_sync(0xffffffffu, bs, o);
      if (v2 < bv || (v2 == bv && s2 < bs)) { bv = v2; bs = s2; }
    }
    if (lane == 0) {
      if (bv < INFINITY) {
        int s = bs;
        #pragma unroll 1
        for (int f = F - 1; f >= 0; --f) { const int Tc = choice[f * smax + s]; newT[f] = (uint8_t)Tc; s -= incT[Tc]; }
      } else {
        #pragma unroll 1
        for (int f = 0; f < F; ++f) newT[f] = oldT[f];
      }
    }
    __syncwarp();
    // ---- apply: pods of the k nodes, then the nearest pod of every source of the functions that use them ---------
    #pragma unroll 1
    for (int f = 0; f < F; ++f) {
      const int nt_ = newT[f], ot_ = oldT[f];
      if (nt_ != ot_) {
        dirtyF |= F <= 64 ? 1ull << f : ~0ull;
        if (lane < kk) c[f * N + Jn[lane]] = (nt_ >> lane) & 1;
        __syncwarp();
        rebuild_pods(f);
      }
      if (nt_ == 0) continue;
      double pj[KK];
#pragma unroll
      for (int q = 0; q < KK; ++q) pj[q] = q < kk ? lam[Jr[q]] * r[f * N + Jr[q]] : kLnsBig;
      #pragma unroll 1
      for (int ib = 0; ib < N; ib += 32) {
        const int i = ib + lane;
        if (i >= N) continue;
        double best = (double)bestv[f * N + i]; int bj = asg[f * N + i];
#pragma unroll
        for (int q = 0; q < KK; ++q) {
          if (q < kk && ((nt_ >> q) & 1)) { const double v = dT[(dix_t)Jr[q] * N + i] + pj[q]; if (v < best || (v == best && Jr[q] < bj)) { best = v; bj = Jr[q]; } }
        }
        bestv[f * N + i] = (float)best; asg[f * N + i] = (pod_t)bj;
      }
    }
    __syncwarp();
  }
  if (lane == 0) {
    const int64_t o = (int64_t)b * 2 * a.chains + chain;
    a.out_g[o] = bestu < INFINITY ? a_d * bestu : INFINITY;
    a.out_g[o + a.chains] = bestg2 < INFINITY ? a_d * bestg2 : INFINITY;
    if (a.out_lb) { a.out_lb[o] = bestu < INFINITY ? a_d * bestg : -INFINITY; a.out_lb[o + a.chains] = bestg2 < INFINITY ? a_d * bestu2 : INFINITY; }
    a.out_round[o] = best_round; a.out_round[o + a.chains] = best_round2;
  }
  if (best_round < 0) for (int q = lane; q < fn; q += 32) outc[q] = c[q];
  if (best_round2 < 0) for (int q = lane; q < fn; q += 32) outc2[q] = c[q];
  if constexpr (St::kGlobal) {
    if (best_round < 0) for (int q = lane; q < fn; q += 32) outa[q] = asg[q];
    if (best_round2 < 0) for (int q = lane; q < fn; q += 32) outa2[q] = asg[q];
  }
