// The body of ball_query_kernel and ball_query_batch_kernel, included into both.  It reads what each kernel
// declares: new_xyz (B,m,3), xyz, B, m, radius, nsample, idx (B,m,nsample), and the macro GF_BQ_SCENE, which declares
// scene b's points P (N,3) and, where the kernel has no N of its own, N.  Indices are local to the scene.  Kept as
// one text so that both kernels search the same way and the single-scene kernel compiles exactly as it did when it
// was written out in place.

  __shared__ float4 sp[BQ_TILE];  // one 16-byte load per candidate
  __shared__ int s_cnt[BQ_CENTRES][BQ_WPC], s_first[BQ_CENTRES][BQ_WPC];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cl = warp / BQ_WPC, part = warp % BQ_WPC;  // centre slot of the CTA, quarter of the tile
  const int groups_per_batch = (m + BQ_CENTRES - 1) / BQ_CENTRES;
  const float r2 = __fmul_rn(radius, radius);
  for (int g = blockIdx.x; g < B * groups_per_batch; g += gridDim.x) {
    const int b = g / groups_per_batch;
    const int j = (g - b * groups_per_batch) * BQ_CENTRES + cl;
    const bool live = j < m;
    GF_BQ_SCENE
    float cx = 0.f, cy = 0.f, cz = 0.f;
    int *row = nullptr;
    if (live) {
      const float *c = new_xyz + ((long long)b * m + j) * 3;
      cx = c[0], cy = c[1], cz = c[2];
      row = idx + ((long long)b * m + j) * nsample;
    }
    int cnt = 0, first = -1;  // hits of this centre so far (same value in its four warps), its first hit
    bool done = !live;
    for (int base = 0; base < N; base += BQ_TILE) {
      const int tn = min(BQ_TILE, N - base);
      __syncthreads();  // previous tile fully consumed
      for (int t = threadIdx.x; t < tn; t += blockDim.x) {  // one point per thread and pass: no index arithmetic
        const float *q = P + ((long long)base + t) * 3;
        sp[t] = make_float4(__ldg(q), __ldg(q + 1), __ldg(q + 2), 0.f);
      }
      __syncthreads();
      unsigned ball[BQ_STEPS];
      int mine = 0, myfirst = -1;
      if (!done) {
#pragma unroll
        for (int u = 0; u < BQ_STEPS; ++u) {
          const int t = part * BQ_PART + 32 * u + lane;
          bool hit = false;
          if (t < tn) {
            const float4 c = sp[t];
            hit = sq3(cx - c.x, cy - c.y, cz - c.z) < r2;
          }
          ball[u] = __ballot_sync(0xffffffffu, hit);
        }
#pragma unroll
        for (int u = 0; u < BQ_STEPS; ++u) mine += __popc(ball[u]);
        if (first < 0 && mine > 0) {  // the centre's first hit is only needed once
#pragma unroll
          for (int u = BQ_STEPS - 1; u >= 0; --u)
            if (ball[u]) myfirst = base + part * BQ_PART + 32 * u + __ffs(ball[u]) - 1;
        }
      }
      if (lane == 0) s_cnt[cl][part] = mine, s_first[cl][part] = myfirst;
      __syncthreads();
      if (!done) {
        int before = cnt;  // hits of the earlier quarters of this tile come first
#pragma unroll
        for (int q = 0; q < BQ_WPC; ++q) {
          const int c = s_cnt[cl][q];
          if (first < 0 && c > 0) first = s_first[cl][q];
          if (q < part) before += c;
          cnt += c;
        }
        if (mine > 0 && before < nsample) {
#pragma unroll
          for (int u = 0; u < BQ_STEPS; ++u) {
            const int pos = before + __popc(ball[u] & ((1u << lane) - 1u));
            if (((ball[u] >> lane) & 1u) && pos < nsample) row[pos] = base + part * BQ_PART + 32 * u + lane;
            before += __popc(ball[u]);
          }
        }
        if (cnt >= nsample) done = true;
      }
      if (__syncthreads_and(done)) break;
    }
    if (live && part == 0) {
      if (cnt > nsample) cnt = nsample;
      const int fill = cnt > 0 ? first : 0;  // ball_query.cpp:22-24 zero-init when nothing is in range
      for (int l = cnt + lane; l < nsample; l += 32) row[l] = fill;
    }
  }
