// The round loop of fps_cluster_kernel and fps_cluster_batch_kernel, included into both kernels' bodies.  It reads
// what each kernel's prologue declares: the template parameters T and P, cluster, CS, crank and scene, the scene's
// xyz (N,3), N, m, L (the reference's block exponent), its output row idx (m), and temp_all (running minima of the
// streaming variant P == 0, one N-float row per scene).  Kept as one text so that both kernels run the same rounds
// and the single-scene kernel compiles exactly as it did when it was written out in place.

  __shared__ FpsSlot slots[2][FPS_MAX_CLUSTER];
  __shared__ uint32_t wkey_v[2][32], wkey_lo[2][32];  // by round parity: no CTA barrier closes a round
  __shared__ __align__(8) uint64_t round_bar[2];  // by round parity: CS x 32 transaction bytes per phase

  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned u = crank * T + tid;  // thread id inside the cluster
  const unsigned bs = 1u << L;
  const unsigned c = u & (bs - 1), g = u >> L;
  const unsigned G = (CS * T) >> L;
  const uint32_t rank_hi = L ? (brev_bits(c, L) << (32 - L)) : 0u;

  constexpr int PR = P > 0 ? P : 1;
  // Points that can never be selected (padding, or |p|^2 <= 1e-3: sampling_gpu.cu:103-104) carry the
  // sentinel running minimum -1: fminf(d, -1) stays -1 and never beats `best`, which starts at -1
  // (the reference's initial value, :93) -- no per-point predicate in the round loop.
  float px[PR], py[PR], pz[PR], tmp[PR];
  if (P > 0) {
#pragma unroll
    for (int i = 0; i < PR; ++i) {
      unsigned k = c + bs * (g * PR + i);
      px[i] = py[i] = pz[i] = 0.f;
      tmp[i] = -1.f;
      if (k < (unsigned)N) {
        px[i] = __ldg(xyz + (size_t)k * 3 + 0);
        py[i] = __ldg(xyz + (size_t)k * 3 + 1);
        pz[i] = __ldg(xyz + (size_t)k * 3 + 2);
        float mag = sq3(px[i], py[i], pz[i]);
        if (!((double)mag <= 1e-3)) tmp[i] = 1e10f;  // eligible: sampling.cpp:74-76
      }
    }
  }
  float *__restrict__ temp = nullptr;
  if (P == 0) {
    temp = temp_all + (size_t)scene * N;
    for (unsigned k = u; k < (unsigned)N; k += CS * T) temp[k] = 1e10f;
  }

  int old = 0;
  float cx = __ldg(xyz + 0), cy = __ldg(xyz + 1), cz = __ldg(xyz + 2);
  if (u == 0) idx[0] = 0;
  if (tid == 0) {
    mbar_init(&round_bar[0], 1);
    mbar_init(&round_bar[1], 1);
    mbar_fence_init();
  }
  cluster.sync();  // barriers initialised everywhere; temp initialised (streaming variant)

  for (int j = 1; j < m; ++j) {
    float best = -1.f;
    uint32_t besti = 0;
    float bx = 0.f, by = 0.f, bz = 0.f;
    if (P > 0) {
#pragma unroll
      for (int i = 0; i < PR; ++i) {
        float d = sq3(px[i] - cx, py[i] - cy, pz[i] - cz);
        float t = fminf(d, tmp[i]);
        tmp[i] = t;
        if (t > best) {
          best = t;
          besti = i;
        }
      }
    } else {
      uint32_t i = 0;
      for (unsigned k = c + bs * g; k < (unsigned)N; k += bs * G, ++i) {
        float x = __ldg(xyz + (size_t)k * 3 + 0), y = __ldg(xyz + (size_t)k * 3 + 1), z = __ldg(xyz + (size_t)k * 3 + 2);
        float mag = sq3(x, y, z);
        if ((double)mag <= 1e-3) continue;
        float d = sq3(x - cx, y - cy, z - cz);
        float t = fminf(d, temp[k]);
        temp[k] = t;
        if (t > best) {
          best = t;
          besti = g + G * i;
          bx = x, by = y, bz = z;
        }
      }
    }
    const bool has = best >= 0.f;
    const uint32_t vb = has ? __float_as_uint(best) : 0u;
    const uint32_t rank = rank_hi | (P > 0 ? (g * PR + besti) : besti);
    const uint32_t lo = has ? ~rank : 0u;

    // warp -> CTA reduction of the 64-bit key with two 32-bit REDUX steps each
    uint32_t wv = __reduce_max_sync(0xffffffffu, vb);
    uint32_t wl = __reduce_max_sync(0xffffffffu, vb == wv ? lo : 0u);
    if (lane == 0) {
      wkey_v[j & 1][warp] = wv;
      wkey_lo[j & 1][warp] = wl;
    }
    // this CTA's own arrival for the round (posted before its candidate can leave, i.e. before any
    // other CTA can run ahead into the next use of this barrier)
    if (tid == 0) mbar_arrive_expect_tx(&round_bar[j & 1], CS * (uint32_t)sizeof(FpsSlot));
    __syncthreads();
    uint32_t tv = lane < T / 32 ? wkey_v[j & 1][lane] : 0u;
    uint32_t tl = lane < T / 32 ? wkey_lo[j & 1][lane] : 0u;
    const uint32_t cv = __reduce_max_sync(0xffffffffu, tv);
    const uint32_t cl = __reduce_max_sync(0xffffffffu, tv == cv ? tl : 0u);

    const int buf = j & 1;
    const bool owner = has && vb == cv && lo == cl;
    const bool nobody = (cv | cl) == 0u;
    // The warp that holds the CTA winner (warp 0 when the CTA has no eligible point) pushes the
    // candidate into every CTA of the cluster: lane r stores it into CTA r's slot with st.async, which
    // completes the transaction bytes of CTA r's round barrier when the data has landed.
    const unsigned own_mask = __ballot_sync(0xffffffffu, owner);
    if (own_mask || (nobody && warp == 0)) {
      const int src = own_mask ? __ffs(own_mask) - 1 : 0;
      if (P > 0 && owner) {
#pragma unroll
        for (int i = 0; i < PR; ++i)
          if (besti == (uint32_t)i) bx = px[i], by = py[i], bz = pz[i];
      }
      const float sx = __shfl_sync(0xffffffffu, bx, src), sy = __shfl_sync(0xffffffffu, by, src),
                  sz = __shfl_sync(0xffffffffu, bz, src);
      if (lane < CS) {
        const uint32_t dst = map_to_cta(smem_u32(&slots[buf][crank]), lane);
        const uint32_t rbar = map_to_cta(smem_u32(&round_bar[buf]), lane);
        st_async_v4(dst, rbar, cv, cl, __float_as_uint(sx), __float_as_uint(sy));
        st_async_v4(dst + 16, rbar, __float_as_uint(sz), 0u, 0u, 0u);
      }
    }
    // round j is use number (j-1)/2 of barrier j&1 (rounds start at 1): wait for that phase
    mbar_wait(&round_bar[buf], (uint32_t)(((j - 1) >> 1) & 1));  // all CS candidates have landed in slots[buf]

    // lane r looks at CTA r's candidate; two REDUX steps pick the cluster-wide winner
    uint32_t sv = 0, sl = 0;
    if (lane < CS) sv = slots[buf][lane].v, sl = slots[buf][lane].lo;
    const uint32_t gv = __reduce_max_sync(0xffffffffu, sv);
    const uint32_t gl = __reduce_max_sync(0xffffffffu, sv == gv ? sl : 0u);
    const unsigned wl_mask = __ballot_sync(0xffffffffu, lane < CS && sv == gv && sl == gl);
    const int wr = __ffs(wl_mask) - 1;  // (gv,gl) != 0 -> exactly one lane; == 0 -> unused
    float nx = 0.f, ny = 0.f, nz = 0.f;
    if (wr >= 0) {
      const FpsSlot &ws = slots[buf][wr];
      nx = ws.x, ny = ws.y, nz = ws.z;
    }
    if ((gv | gl) == 0u) {  // no eligible point anywhere: the reference's tree yields index 0
      old = 0;
      cx = __ldg(xyz + 0), cy = __ldg(xyz + 1), cz = __ldg(xyz + 2);
    } else {
      uint32_t rk = ~gl;
      old = L ? (int)(((rk & ((1u << (32 - L)) - 1u)) << L) | brev_bits(rk >> (32 - L), L)) : (int)rk;
      cx = nx, cy = ny, cz = nz;
    }
    if (u == 0) idx[j] = old;
  }
