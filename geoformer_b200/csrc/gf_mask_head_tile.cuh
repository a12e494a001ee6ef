// The body of one 128-point tile of mask_head_kernel and mask_head_batch_kernel, included into both inside their tile
// loops.  It reads what each kernel declares: `a` (MhArgs of the tile's scene: geo, feats, coords, out, dlogit, dfeats
// and the constants mh_stage_group reads, N and Q), `tile` (the tile's index within its scene), G, `it` (the running
// count of query groups issued by this CTA), `part` (the partial sums this tile adds to; backward) and `first_tile`
// (the tile starts those partial sums).  Kept as one text so that both kernels compute every logit and gradient the
// same way and the single-scene kernel compiles exactly as it did when it was written out in place.
    const int p = (int)(lq * 32u + lane), n = tile * MH_TILE + p;
    const bool valid = n < a.N;
    {  // feats tile: row = point (zero past N), 16 channels of the 32-float swizzled row
      const int r = (int)(tid >> 2), c0 = (int)(tid & 3u) * 4, nr = tile * MH_TILE + r;
      float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
      if (nr < a.N) {
        const float *src = a.feats + (size_t)nr * MH_M + c0;
        f = make_float4(__ldg(src), __ldg(src + 1), __ldg(src + 2), __ldg(src + 3));
      }
      *reinterpret_cast<float4 *>(sA + sw128_off<MH_TILE>(r, c0)) = f;
    }
    const float px = valid ? __ldg(a.coords + (size_t)n * 3 + 0) : 0.f, py = valid ? __ldg(a.coords + (size_t)n * 3 + 1) : 0.f,
                pz = valid ? __ldg(a.coords + (size_t)n * 3 + 2) : 0.f;
    float fx[BWD ? MH_M : 1], dfa[BWD ? MH_M : 1];
    if (BWD) {
#pragma unroll
      for (int c = 0; c < MH_M; ++c) {
        fx[c] = valid ? __ldg(a.feats + (size_t)n * MH_M + c) : 0.f;
        dfa[c] = 0.f;
      }
    }
    mh_stage_group(a, 0, sB + (it & 1u) * MH_B_BYTES, reinterpret_cast<MhConst *>(sCraw + (it & 1u) * MH_C_BYTES), tid);
    mh_sync_for_mma();
    if (tid == 0) issue(it);

    for (int g = 0; g < G; ++g) {
      const uint32_t cur = it + (uint32_t)g, buf = cur & 1u;
      // map entries (and upstream gradients) of this warp's 4 queries, in flight while the product runs
      float gv[4], dl[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int q = g * MH_QG + (int)qq * 4 + i;
        const bool live = valid && q < a.Q;
        gv[i] = live ? __ldg(a.geo + (size_t)q * a.N + n) : 0.f;
        dl[i] = BWD && live ? __ldg(a.dlogit + (size_t)q * a.N + n) : 0.f;
      }
      if (g + 1 < G) {
        mh_stage_group(a, g + 1, sB + (buf ^ 1u) * MH_B_BYTES, reinterpret_cast<MhConst *>(sCraw + (buf ^ 1u) * MH_C_BYTES), tid);
        mh_sync_for_mma();
        if (tid == 0) issue(cur + 1);
      }
      mbar_wait(buf ? mbar1 : mbar0, (cur >> 1) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const MhConst *sc = reinterpret_cast<const MhConst *>(sCraw + buf * MH_C_BYTES);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ql = (int)qq * 4 + i, q = g * MH_QG + ql;
        float d[16];
        tmem_ld16(t_lane + buf * MH_COLS + (uint32_t)i * 16u, d);  // every lane: .sync.aligned
        if (q >= a.Q) continue;  // warp-uniform
        const float4 sd = sc->seed[ql];
        const bool un = gv[i] < 0.f;
        const float r0 = mask_push(__fsub_rn(sd.x, px), sd.w, un), r1 = mask_push(__fsub_rn(sd.y, py), sd.w, un),
                    r2 = mask_push(__fsub_rn(sd.z, pz), sd.w, un);
        if (!BWD) {
          float o = sc->b1[ql];
#pragma unroll
          for (int j = 0; j < MH_M; ++j) {
            const int col = ql * MH_M + j;
            o = __fmaf_rn(sc->w1[col], mh_relu(mh_hidden(d[j], sc->wr[col], r0, r1, r2)), o);
          }
          if (valid) __stcs(a.out + (size_t)q * a.N + n, o);
        } else {
          const float gl = dl[i];
          float grh[MH_M], dh[MH_M];
#pragma unroll
          for (int j = 0; j < MH_M; ++j) {
            const int col = ql * MH_M + j;
            const float h = mh_hidden(d[j], sc->wr[col], r0, r1, r2);
            grh[j] = __fmul_rn(gl, mh_relu(h));
            dh[j] = h <= 0.f ? 0.f : __fmul_rn(gl, sc->w1[col]);  // torch's ReLU backward: a NaN h passes g
          }
          float *dst = sPart + ((size_t)lq * MH_QG + ql) * MH_NPART;
          // dw1, db0, dw0 coordinate part (and db1): four channels j per 32-value chunk
#pragma unroll
          for (int j4 = 0; j4 < MH_M; j4 += 4) {
            float v[32];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const float x = dh[j4 + jj];
              v[jj * 8 + 0] = grh[j4 + jj];
              v[jj * 8 + 1] = x;
              v[jj * 8 + 2] = __fmul_rn(x, r0);
              v[jj * 8 + 3] = __fmul_rn(x, r1);
              v[jj * 8 + 4] = __fmul_rn(x, r2);
              v[jj * 8 + 5] = (j4 + jj == 0) ? gl : 0.f;
              v[jj * 8 + 6] = 0.f;
              v[jj * 8 + 7] = 0.f;
            }
            dst[256 + j4 * 8 + lane] = mh_warp_reduce32(v, lane);
          }
          // dw0 feature part: two channels j per chunk; dfeats += dh w0f in fixed (q, j) order
#pragma unroll
          for (int jp = 0; jp < MH_M; jp += 2) {
            float v[32];
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
              const int row = ql * MH_M + jp + jj;
#pragma unroll
              for (int c4 = 0; c4 < MH_M; c4 += 4) {
                const float4 w = *reinterpret_cast<const float4 *>(sB + buf * MH_B_BYTES + sw128_off<MH_COLS>(row, c4));
                dfa[c4 + 0] = __fmaf_rn(dh[jp + jj], w.x, dfa[c4 + 0]);
                dfa[c4 + 1] = __fmaf_rn(dh[jp + jj], w.y, dfa[c4 + 1]);
                dfa[c4 + 2] = __fmaf_rn(dh[jp + jj], w.z, dfa[c4 + 2]);
                dfa[c4 + 3] = __fmaf_rn(dh[jp + jj], w.w, dfa[c4 + 3]);
              }
#pragma unroll
              for (int c = 0; c < MH_M; ++c) v[jj * 16 + c] = __fmul_rn(dh[jp + jj], fx[c]);
            }
            dst[jp * 16 + lane] = mh_warp_reduce32(v, lane);
          }
        }
      }
      // TMEM buffer, constants (and partial sums) of this group are free once every thread is past this point
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();
      if (BWD) {  // the tile's sums over its four lane quarters, added to this CTA's partials in tile order
        for (int e = (int)tid; e < MH_QG * MH_NPART; e += MH_THREADS) {
          const int ql = e / MH_NPART, q = g * MH_QG + ql;
          if (q >= a.Q) continue;
          float s = sPart[e];
          s = __fadd_rn(s, sPart[MH_QG * MH_NPART + e]);
          s = __fadd_rn(s, sPart[2 * MH_QG * MH_NPART + e]);
          s = __fadd_rn(s, sPart[3 * MH_QG * MH_NPART + e]);
          float *pp = part + (size_t)g * MH_QG * MH_NPART + e;
          *pp = first_tile ? s : __fadd_rn(*pp, s);
        }
        __syncthreads();
      }
    }
    it += (uint32_t)G;
    if (BWD) {  // dfeats of the tile: the four query quarters summed in order
      float *sD = sPart;
#pragma unroll
      for (int c = 0; c < MH_M; ++c) sD[((size_t)qq * MH_TILE + p) * MH_M + c] = dfa[c];
      __syncthreads();
      for (int e = (int)tid; e < MH_TILE * MH_M; e += MH_THREADS) {
        const int pr = e / MH_M, nr = tile * MH_TILE + pr;
        if (nr >= a.N) continue;
        float s = sD[e];
        s = __fadd_rn(s, sD[MH_TILE * MH_M + e]);
        s = __fadd_rn(s, sD[2 * MH_TILE * MH_M + e]);
        s = __fadd_rn(s, sD[3 * MH_TILE * MH_M + e]);
        a.dfeats[(size_t)nr * MH_M + (e - pr * MH_M)] = s;
      }
      __syncthreads();
    }
    first_tile = false;
