// The round loop of fps_cluster_kernel and fps_cluster_batch_kernel, included into both kernels' bodies.  It reads
// what each kernel's prologue declares: the template parameters T and P (P > 0 points per thread, held in registers),
// cluster, CS and crank, the scene's xyz (N,3), N, m, L (the reference's block exponent) and its output row idx (m).
// Kept as one text so that both kernels run the same rounds and the single-scene kernel compiles exactly as it did
// when it was written out in place.

  __shared__ FpsSlot slots[2][FPS_MAX_CLUSTER];
  __shared__ uint32_t wkey_v[2][32], wkey_lo[2][32];  // by round parity: no CTA barrier closes a round
  __shared__ __align__(8) uint64_t round_bar[2];  // by round parity: CS x 32 transaction bytes per phase

  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned u = crank * T + tid;  // thread id inside the cluster
  const unsigned bs = 1u << L;
  const unsigned c = u & (bs - 1), g = u >> L;
  const uint32_t rank_hi = fps_rank_hi(c, L);

  // Points that can never be selected (padding, or not fps_eligible) carry the sentinel running minimum -1:
  // fminf(d, -1) stays -1 and never beats `best`, which starts at -1 (the reference's initial value,
  // sampling_gpu.cu:93) -- no per-point predicate in the round loop.
  float px[P], py[P], pz[P], tmp[P];
#pragma unroll
  for (int i = 0; i < P; ++i) {
    unsigned k = c + bs * (g * P + i);
    px[i] = py[i] = pz[i] = 0.f;
    tmp[i] = -1.f;
    if (k < (unsigned)N) {
      px[i] = __ldg(xyz + (size_t)k * 3 + 0);
      py[i] = __ldg(xyz + (size_t)k * 3 + 1);
      pz[i] = __ldg(xyz + (size_t)k * 3 + 2);
      if (fps_eligible(px[i], py[i], pz[i])) tmp[i] = 1e10f;
    }
  }

  float cx = __ldg(xyz + 0), cy = __ldg(xyz + 1), cz = __ldg(xyz + 2);
  if (u == 0) idx[0] = 0;
  if (tid == 0) {
    mbar_init(&round_bar[0], 1);
    mbar_init(&round_bar[1], 1);
    mbar_fence_init();
  }
  cluster.sync();  // barriers initialised everywhere

  for (int j = 1; j < m; ++j) {
    float best = -1.f;
    uint32_t besti = 0;
    float bx = 0.f, by = 0.f, bz = 0.f;
#pragma unroll
    for (int i = 0; i < P; ++i) {
      float d = sq3(px[i] - cx, py[i] - cy, pz[i] - cz);
      float t = fminf(d, tmp[i]);
      tmp[i] = t;
      if (t > best) {
        best = t;
        besti = i;
      }
    }
    const bool has = best >= 0.f;
    const FpsKey key = {has ? __float_as_uint(best) : 0u, has ? ~(rank_hi | (g * P + besti)) : 0u};

    // warp -> CTA reduction of the 64-bit key
    const FpsKey wk = warp_max(key);
    if (lane == 0) {
      wkey_v[j & 1][warp] = wk.v;
      wkey_lo[j & 1][warp] = wk.lo;
    }
    // this CTA's own arrival for the round (posted before its candidate can leave, i.e. before any
    // other CTA can run ahead into the next use of this barrier)
    if (tid == 0) mbar_arrive_expect_tx(&round_bar[j & 1], CS * (uint32_t)sizeof(FpsSlot));
    __syncthreads();
    const FpsKey ck = warp_max({lane < T / 32 ? wkey_v[j & 1][lane] : 0u, lane < T / 32 ? wkey_lo[j & 1][lane] : 0u});

    const int buf = j & 1;
    // field by field: `has && key == ck` allocates the kernel's registers differently
    const bool owner = has && key.v == ck.v && key.lo == ck.lo;
    const bool nobody = (ck.v | ck.lo) == 0u;
    // The warp that holds the CTA winner (warp 0 when the CTA has no eligible point) pushes the
    // candidate into every CTA of the cluster: lane r stores it into CTA r's slot with st.async, which
    // completes the transaction bytes of CTA r's round barrier when the data has landed.
    const unsigned own_mask = __ballot_sync(0xffffffffu, owner);
    if (own_mask || (nobody && warp == 0)) {
      const int src = own_mask ? __ffs(own_mask) - 1 : 0;
      if (owner) {
#pragma unroll
        for (int i = 0; i < P; ++i)
          if (besti == (uint32_t)i) bx = px[i], by = py[i], bz = pz[i];
      }
      const float sx = __shfl_sync(0xffffffffu, bx, src), sy = __shfl_sync(0xffffffffu, by, src),
                  sz = __shfl_sync(0xffffffffu, bz, src);
      if (lane < CS) {
        const uint32_t dst = map_to_cta(smem_u32(&slots[buf][crank]), lane);
        const uint32_t rbar = map_to_cta(smem_u32(&round_bar[buf]), lane);
        st_async_v4(dst, rbar, ck.v, ck.lo, __float_as_uint(sx), __float_as_uint(sy));
        st_async_v4(dst + 16, rbar, __float_as_uint(sz), 0u, 0u, 0u);
      }
    }
    // round j is use number (j-1)/2 of barrier j&1 (rounds start at 1): wait for that phase
    mbar_wait(&round_bar[buf], (uint32_t)(((j - 1) >> 1) & 1));  // all CS candidates have landed in slots[buf]

    // lane r looks at CTA r's candidate; two REDUX steps pick the cluster-wide winner
    FpsKey sk = {0u, 0u};
    if (lane < CS) sk = {slots[buf][lane].v, slots[buf][lane].lo};
    const FpsKey gk = warp_max(sk);
    const unsigned wl_mask = __ballot_sync(0xffffffffu, lane < CS && sk.v == gk.v && sk.lo == gk.lo);
    const int wr = __ffs(wl_mask) - 1;  // gk != 0 -> exactly one lane; gk == 0 -> unused
    float nx = 0.f, ny = 0.f, nz = 0.f;
    if (wr >= 0) {
      const FpsSlot &ws = slots[buf][wr];
      nx = ws.x, ny = ws.y, nz = ws.z;
    }
    const int old = fps_round_end(gk, nx, ny, nz, xyz, L, cx, cy, cz);
    if (u == 0) idx[j] = old;
  }
