// gemm_tc_kernel.cuh — the body of the tensor-core GEMM kernel (gemm_tc.cu), compiled twice: as gemm_tc_kernel (every shape
// whose output width is a multiple of the tile width) and as gemm_tc_tail_kernel (VITB_TC_TAIL, output width 64 mod 128).
// Included by gemm_tc.cu only, with VITB_TC_KERNEL and VITB_TC_TAIL defined.
// TAIL (fwd / dgrad whose output width is 64 mod 128): the last column block is a partial tile.  TMA zero-fills the operand
// rows / columns past the edge (the full box still counts towards the barrier's transaction bytes) and clips the stores; the
// only per-thread reads of the epilogue, bias and pos_emb, skip the 64-column slabs at or past p.valid_n.
template <int BN, bool A_MN, bool B_MN, int NS, int STAGES, int KPS, int NSLAB, bool W_RES, int CG, bool DROP>
__global__ void __launch_bounds__(tc_threads(NS, epi_warps_for(BN, NSLAB)), 1)
    VITB_TC_KERNEL(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                   const __grid_constant__ CUtensorMap tma_out, const __grid_constant__ CUtensorMap tma_pre,
                   const __grid_constant__ CUtensorMap tma_in, const TcArgs p) {
  constexpr bool TAIL = VITB_TC_TAIL;
  using S = TcSmem<BN, NS, STAGES, KPS, NSLAB, W_RES, CG>;
  constexpr int ACC = S::kAcc;
  constexpr int EW = S::kEW;
  constexpr bool PAIR = CG == 2;
  static_assert(!PAIR || (W_RES && !A_MN && NSLAB > 0 && KPS == 1), "pair mode: resident-weight fwd / dgrad kernels only");
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
  const bool is_leader = cta_rank == 0;
  static_assert(NS * ACC * BN + NS * 16 <= (int)kTmemCols || NSLAB > 0, "TMEM plan");
  static_assert(BN == 128 || (BN == 192 && NSLAB > 0 && !W_RES && CG == 1) || (NSLAB == 0 && BN % 64 == 0 && BN <= 256),
                "slab epilogue: one warp per TMEM lane quarter and 64-column group (BN = 128: 8 warps, BN = 192: 12); the fp32 direct-store epilogue takes any BN = 64 j");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  pdl_trigger();

  // st = stream, s = ring stage, j = k-block inside the stage
  auto a_stage = [&](int st, int s, int j) {
    return smem_base + S::kRingOff + (uint32_t)st * S::kRingBytes + (uint32_t)s * S::kStageBytes + (uint32_t)j * S::kSubBytes;
  };
  auto b_stage = [&](int st, int s, int j) { return a_stage(st, s, j) + S::kABytes; };
  auto b_res = [&](int kb) { return smem_base + (uint32_t)kb * S::kBBytes; };  // W_RES: resident k-block kb of B
  const uint32_t epi_base = smem_base + S::kEpiOff;
  const uint32_t bar_base = smem_base + S::kBarOff;
  auto full_bar = [&](int st, int s) { return bar_base + (uint32_t)(st * S::kBarsPerStream + s) * 8; };
  auto empty_bar = [&](int st, int s) { return bar_base + (uint32_t)(st * S::kBarsPerStream + STAGES + s) * 8; };
  auto tfull_bar = [&](int st, int a) { return bar_base + (uint32_t)(st * S::kBarsPerStream + 2 * STAGES + a) * 8; };
  auto tempty_bar = [&](int st, int a) { return bar_base + (uint32_t)(st * S::kBarsPerStream + 2 * STAGES + 2 + a) * 8; };
  auto in_bar = [&](int w) { return bar_base + (uint32_t)(NS * S::kBarsPerStream + w) * 8; };
  const uint32_t wfull_bar = bar_base + (uint32_t)(NS * S::kBarsPerStream + EW) * 8;
  // TMEM columns: accumulator a of stream st, and the stream's 16-column bias-gradient accumulator (wgrad)
  auto acc_col = [&](int st, int a) { return (uint32_t)((st * ACC + a) * BN); };
  auto bias_col = [&](int st, int a) { return (uint32_t)(NS * ACC * BN + (st * ACC + a) * 16); };
  const uint32_t tmem_slot = bar_base + S::kNumBars * 8;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + S::kBarOff + S::kNumBars * 8);

  const bool want_dbias = (p.e.mode == EPI_RAW_F32) && (p.dbias_part != nullptr);

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_b) : "memory");
    if (p.e.mode != EPI_RAW_F32) asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_out) : "memory");
    for (int st = 0; st < NS; ++st) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(full_bar(st, s), 1);
        mbar_init(empty_bar(st, s), 1);
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(tfull_bar(st, a), 1);
        mbar_init(tempty_bar(st, a), EW * CG);  // one arrival per epilogue warp (of both CTAs of a pair)
      }
    }
    for (int w = 0; w < EW; ++w) mbar_init(in_bar(w), 1);
    mbar_init(wfull_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == NS) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  if (want_dbias && warp >= 2 * NS) {
    // all-ones bf16 operand (16 rows x 128 B, any layout reads ones); overlays the unused epilogue slabs
    uint32_t* ones = reinterpret_cast<uint32_t*>(smem_gen + S::kEpiOff);
    for (int i = threadIdx.x - 64 * NS; i < 2048 / 4; i += EW * 32) ones[i] = 0x3F803F80u;
    fence_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();  // the peer's barriers exist before anything is signalled remotely
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  // everything above (barriers, TMEM allocation, tensor-map prefetch, the ones operand) overlapped the previous kernel's tail;
  // operands, residuals and outputs may belong to it: wait for it here
  pdl_wait();

  const int tiles_per_split = p.num_m_blocks * p.num_n_blocks;
  const int num_tiles = tiles_per_split * p.splits;
  // work decomposition.  streaming: tile = blockIdx.x + it * gridDim.x over (split, m-block, n-block), n fastest.
  // W_RES: CTA = (n-block group, member); member walks m-blocks member, member + members, ...
  // (pair mode: the unit is the CTA pair, p.num_m_blocks counts 256-row blocks)
  const int res_groups = p.num_n_blocks;
  const int unit = (int)blockIdx.x / CG, units = (int)gridDim.x / CG;
  const int res_members = W_RES ? units / res_groups : 1;
  const int res_group = W_RES ? unit % res_groups : 0;
  const int res_member = W_RES ? unit / res_groups : 0;
  const bool res_active = !W_RES || res_member < res_members;
  auto get_tile = [&](int it, int& m0, int& n0, int& nblk, int& split) -> bool {
    if (W_RES) {
      const int mb = res_member + it * res_members;
      if (!res_active || mb >= p.num_m_blocks) return false;
      m0 = (mb * CG + (int)cta_rank) * BM; nblk = res_group; n0 = nblk * BN; split = 0;
      return true;
    }
    const int tile = (int)blockIdx.x + it * (int)gridDim.x;
    if (tile >= num_tiles) return false;
    split = tile / tiles_per_split;
    const int rem = tile - split * tiles_per_split;
    m0 = (rem / p.num_n_blocks) * BM;
    nblk = rem % p.num_n_blocks;
    n0 = nblk * BN;
    return true;
  };

  if (warp < NS) {
    // ================= TMA producer of stream `warp`: the whole warp walks the loop, one elected lane issues =================
    const int st_ = warp;
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    if (W_RES && res_active && leader && st_ == 0) {  // the weight block of this CTA (its half, in a pair): every k-block, once
      const int n0 = res_group * BN + (int)cta_rank * (BN / CG);
      const uint32_t wbar = PAIR ? mapa_rank(wfull_bar, 0) : wfull_bar;  // the leader's barrier collects both halves
      if (is_leader) mbar_arrive_expect_tx(wfull_bar, (uint32_t)p.kblocks_total * S::kBBytes * CG);
      for (int kb = 0; kb < p.kblocks_total; ++kb) {
        if (!B_MN) {
          if (PAIR) tma_load_2d_pair(b_res(kb), &tma_b, wbar, kb * BK, n0);
          else tma_load_2d(b_res(kb), &tma_b, wfull_bar, kb * BK, n0);
        } else {
#pragma unroll
          for (int j = 0; j < BN / CG / 64; ++j) {
            if (PAIR) tma_load_2d_pair(b_res(kb) + j * (64 * BK * 2), &tma_b, wbar, n0 + j * 64, kb * BK);
            else tma_load_2d(b_res(kb) + j * (64 * BK * 2), &tma_b, wfull_bar, n0 + j * 64, kb * BK);
          }
        }
      }
    }
    __syncwarp();
    int m0, n0, nblk, split;
    for (int it = st_; get_tile(it, m0, n0, nblk, split); it += NS) {
      const int kb0 = split * p.kblocks_per_split;
      const int kb1 = min(p.kblocks_total, kb0 + p.kblocks_per_split);
      if (!A_MN && p.pf_tiles > 0 && leader) {
        // The ring holds < 1 tile of A per stream, HBM latency under load is several tile times: ask L2 for the A rows of a
        // tile further ahead.  Every row block is requested once: resident mode splits the k-blocks over the CTAs that share
        // the row block (one per column block, same pace); streaming mode lets the CTA at column block 0 do it.
        if (W_RES) {
          int pm0, pn0, pnblk, psplit;
          if (get_tile(it + p.pf_tiles * NS, pm0, pn0, pnblk, psplit)) {
            for (int kb = res_group; kb < p.kblocks_total; kb += res_groups) tma_prefetch_2d(&tma_a, kb * BK, pm0);
            if (p.pf_in && p.has_in) {  // the epilogue's input operand (residual / z) of that tile: 64 x 32 boxes
#pragma unroll
              for (int c = 0; c < BN / 64; ++c)
#pragma unroll
                for (int q = 0; q < 4; ++q) tma_prefetch_2d(&tma_in, pn0 + c * 64, pm0 + q * 32);
            }
          }
        } else if (nblk == 0) {
          const int pm0 = m0 + ceil_div_dev(p.pf_tiles * NS * (int)gridDim.x, p.num_n_blocks) * BM;
          if (pm0 < p.num_m_blocks * BM)
            for (int kb = kb0; kb < kb1; ++kb) tma_prefetch_2d(&tma_a, kb * BK, pm0);
        }
      }
      for (int kb = kb0; kb < kb1; kb += KPS) {
        const int nsub = min(KPS, kb1 - kb);
        if (A_MN && p.pf_kblocks > 0 && leader && p.a3_pp == 0) {
          // wgrad: both operands stream from HBM along the reduction; the CTAs of one split share them (A over the column
          // blocks, B over the row blocks), so the one at block 0 of the other dimension prefetches
          const int pk = (kb + p.pf_kblocks) * BK;
          if (kb + p.pf_kblocks < kb1) {
            if (nblk == 0) {
#pragma unroll
              for (int q = 0; q < BM / 64; ++q) tma_prefetch_2d(&tma_a, m0 + q * 64, pk);
            }
            if (m0 == 0) {
#pragma unroll
              for (int q = 0; q < BN / 64; ++q) tma_prefetch_2d(&tma_b, n0 + q * 64, pk);
            }
          }
        }
        mbar_wait(empty_bar(st_, stage), phase ^ 1u);
        // pair mode: the full barrier of the LEADER counts the bytes of both CTAs; the leader arms it, both load
        const uint32_t fbar = PAIR ? mapa_rank(full_bar(st_, stage), 0) : full_bar(st_, stage);
        if (leader && (p.dbg_flags & 2)) {
          mbar_arrive(fbar);
        } else if (leader) {
          if (is_leader) mbar_arrive_expect_tx(full_bar(st_, stage), (uint32_t)nsub * S::kSubBytes * CG);
#pragma unroll
          for (int j = 0; j < KPS; ++j) {
            if (j < nsub) {
              const int k0 = (kb + j) * BK;
              const uint32_t sa = a_stage(st_, stage, j), sb = b_stage(st_, stage, j);
              if (!A_MN) {
                if (PAIR) tma_load_2d_pair(sa, &tma_a, fbar, k0, m0);
                else tma_load_2d(sa, &tma_a, fbar, k0, m0);
              } else if (p.a3_pp > 0) {
                // 64 reduction rows = token rows [a3_off + k0 % pp, +64) of image k0 / pp  (pp >= 64), or all pp token rows of
                // 64 / pp consecutive images (pp < 64); the box of the 3-D map has exactly that shape
                const int img = k0 / p.a3_pp, tok = p.a3_off + (p.a3_pp >= 64 ? k0 % p.a3_pp : 0);
#pragma unroll
                for (int q = 0; q < BM / 64; ++q) tma_load_3d(sa + q * (64 * BK * 2), &tma_a, fbar, m0 + q * 64, tok, img);
              } else {
#pragma unroll
                for (int q = 0; q < BM / 64; ++q) tma_load_2d(sa + q * (64 * BK * 2), &tma_a, fbar, m0 + q * 64, k0);
              }
              if (!W_RES) {
                if (!B_MN) {
                  tma_load_2d(sb, &tma_b, fbar, k0, n0);
                } else {
#pragma unroll
                  for (int q = 0; q < BN / 64; ++q) tma_load_2d(sb + q * (64 * BK * 2), &tma_b, fbar, n0 + q * 64, k0);
                }
              }
            }
          }
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp < 2 * NS) {
    // ================= MMA issuer of stream `warp - NS`: the whole warp walks the loop, one elected lane issues =================
    // (pair mode: only the leader CTA's issuers run; their MMAs drive the tensor cores and TMEM of both SMs)
    const int st_ = warp - NS;
    const bool leader = elect_one() && is_leader;
    // instruction descriptor: D fp32, A/B bf16, majors, N>>3, M>>4
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
                           ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((BM * CG) >> 4) << 24);
    // bias-gradient MMA: same A, B = all-ones K-major tile, N = 16
    const uint32_t idesc_ones = (1u << 4) | (1u << 7) | (1u << 10) | ((A_MN ? 1u : 0u) << 15) | (0u << 16) |
                                ((uint32_t)(16 >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    const uint64_t ones_desc = make_smem_desc(epi_base, 16, 1024);
    // K-major: a k-step is 16 elements (32 B) inside the swizzle atom, LBO unused (16).  MN-major: a k-step is 16 k-rows
    // (2048 B), LBO = distance between 64-wide MN atoms.
    constexpr uint32_t kALbo = A_MN ? BK * 128 : 16, kBLbo = B_MN ? BK * 128 : 16;
    constexpr uint32_t kAStep = (A_MN ? UK * 128 : UK * 2) >> 4, kBStep = (B_MN ? UK * 128 : UK * 2) >> 4;
    const uint32_t a_lo0 = desc_lo(a_stage(st_, 0, 0), kALbo);
    const uint32_t b_lo0 = desc_lo(W_RES ? b_res(0) : b_stage(st_, 0, 0), kBLbo);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    long long t_full = 0, t_tempty = 0, t_issue = 0, t_commit = 0, t_begin = clock64();
    if (W_RES && res_active && is_leader) {
      mbar_wait(wfull_bar, 0);
      tc_fence_after();
    }
    const long long t_w = clock64() - t_begin;
    int m0, n0, nblk, split;
    int ntiles = 0;
    for (int it = st_; is_leader && get_tile(it, m0, n0, nblk, split); it += NS) {
      ++ntiles;
      const bool do_bias = want_dbias && nblk == 0;
      const int kb0 = split * p.kblocks_per_split;
      const int kb1 = min(p.kblocks_total, kb0 + p.kblocks_per_split);
      long long t0 = p.dbg ? clock64() : 0;
      mbar_wait(tempty_bar(st_, acc), acc_phase ^ 1u);
      tc_fence_after();
      if (p.dbg) t_tempty += clock64() - t0;
      const uint32_t d_tmem = tmem_base + acc_col(st_, acc);
      const uint32_t d_bias = tmem_base + bias_col(st_, acc);
      for (int kb = kb0; kb < kb1; kb += KPS) {
        const int nsub = min(KPS, kb1 - kb);
        t0 = p.dbg ? clock64() : 0;
        mbar_wait(full_bar(st_, stage), phase);
        tc_fence_after();
        if (p.dbg) t_full += clock64() - t0;
        if (leader) {
          const long long ti0 = p.dbg ? clock64() : 0;
#pragma unroll
          for (int j = 0; j < KPS; ++j) {
            if (j < nsub) {
              const uint32_t a_lo = a_lo0 + (uint32_t)(stage * KPS + j) * (S::kSubBytes >> 4);
              const uint32_t b_lo = b_lo0 + (W_RES ? (uint32_t)(kb + j) * (S::kBBytes >> 4) : (uint32_t)(stage * KPS + j) * (S::kSubBytes >> 4));
              const uint32_t first = (kb + j) > kb0 ? 1u : 0u;
              if (PAIR) {
#pragma unroll
                for (int kk = 0; kk < BK / UK; ++kk)
                  tc_mma_bf16_pair(d_tmem, desc_from_lo(a_lo + kk * kAStep), desc_from_lo(b_lo + kk * kBStep), idesc, kk > 0 ? 1u : first);
              } else if (!do_bias) {
#pragma unroll
                for (int kk = 0; kk < BK / UK; ++kk)
                  tc_mma_bf16(d_tmem, desc_from_lo(a_lo + kk * kAStep), desc_from_lo(b_lo + kk * kBStep), idesc, kk > 0 ? 1u : first);
              } else {
#pragma unroll
                for (int kk = 0; kk < BK / UK; ++kk) {
                  tc_mma_bf16(d_tmem, desc_from_lo(a_lo + kk * kAStep), desc_from_lo(b_lo + kk * kBStep), idesc, kk > 0 ? 1u : first);
                  tc_mma_bf16(d_bias, desc_from_lo(a_lo + kk * kAStep), ones_desc, idesc_ones, kk > 0 ? 1u : first);
                }
              }
            }
          }
          const long long ti1 = p.dbg ? clock64() : 0;
          if (PAIR) tc_commit_pair(empty_bar(st_, stage));  // frees the slot in both CTAs
          else tc_commit(empty_bar(st_, stage));             // frees the smem slot once these MMAs have read it
          if (p.dbg) { t_issue += ti1 - ti0; t_commit += clock64() - ti1; }
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
      if (leader) {  // accumulator complete
        if (PAIR) tc_commit_pair(tfull_bar(st_, acc));
        else tc_commit(tfull_bar(st_, acc));
      }
      __syncwarp();
      if (++acc == ACC) { acc = 0; acc_phase ^= 1u; }
    }
    if (p.dbg && leader && st_ == 0) {
      long long* d = p.dbg + (size_t)blockIdx.x * 8;
      d[0] = clock64() - t_begin; d[1] = t_full; d[2] = t_tempty; d[3] = t_w; d[4] = ntiles; d[6] = t_issue; d[7] = t_commit;
    }
  } else {
    // ================= epilogue: 8 warps; TMEM lane quarter = warp % 4, column half = ew / 4.  Tiles are drained in
    // the CTA's tile order, alternating between the streams ==========
    const int ew = warp - 2 * NS;
    const int quarter = warp & 3;
    const int half = ew >> 2;                         // column group of this warp: 64 columns in the slab epilogue, BN / 2 in the fp32 one
    constexpr int kColW = NSLAB > 0 ? 64 : BN / 2;
    const int row_in_tile = quarter * 32 + lane;
    // slab 0: output — and, before that, the input operand (residual / z), which is consumed in place; slab 1: pre-activation
    const uint32_t slab_out = epi_base + (uint32_t)(ew * NSLAB + 0) * kSlabBytes;
    const uint32_t slab_pre = epi_base + (uint32_t)(ew * NSLAB + (NSLAB > 1 ? 1 : 0)) * kSlabBytes;
    const uint32_t slab_in = slab_out;
    uint32_t in_phase = 0;
    const EpiParams& e = p.e;
    bool stores_pending = false;
    // (DROP is a template parameter, not only a run-time flag: the mask arithmetic inside the epilogue costs the p = 0 kernels
    // a few spilled registers otherwise)
    const bool dropping = DROP && NSLAB > 0 && p.drop.thr != 0;
    const uint32_t drop_st = dropping ? drop_step(p.drop) : 0u;
    // this thread's 64 values of output row `grow`, columns n0 .. n0 + 63: eight mask groups of the flattened [M, N] output
    auto drop64 = [&](float (&v)[64], int grow, int n0) {
      const uint64_t g0 = ((uint64_t)grow * (uint64_t)p.N + (uint64_t)n0) >> 3;
#pragma unroll
      for (int j = 0; j < 8; ++j) drop_apply8(&v[8 * j], drop_words(p.drop, drop_st, g0 + j), p.drop.thr, p.drop.scale);
    };
    int m0, nb0, nblk, split;
    for (int it = 0; get_tile(it, m0, nb0, nblk, split); ++it) {
      const int st_ = it % NS, jt = it / NS;           // stream, and the tile's index inside the stream
      const int acc = jt % ACC;
      const uint32_t acc_phase = (uint32_t)(jt / ACC) & 1u;
      const int n0 = nb0 + half * kColW;
      const int grow = m0 + row_in_tile;
      if (p.has_in) {  // fetch this warp's residual / z slab while the MMAs of the tile run
        if (lane == 0) {
          if (stores_pending) tma_store_wait_read();  // the slab doubles as the output slab of the previous tile
          mbar_arrive_expect_tx(in_bar(ew), kSlabBytes);
          // (patch embedding: the "residual" is pos_emb, whose row is the token of the GEMM row, not the GEMM row itself)
          const int in_row = p.out3 ? e.rm_offset + (m0 + quarter * 32) % e.rm_group : m0 + quarter * 32;
          tma_load_2d(slab_in, &tma_in, in_bar(ew), n0, in_row);
        }
      }
      // the 64 bias values of this warp's columns (two 128-byte lines): on their way while the tile's MMAs run, so that a
      // single-tile kernel does not add an L2 round trip after its accumulator is ready
      // (TAIL: a 64-column slab lies wholly inside or wholly past the edge)
      if (kBiasPrefetch && NSLAB > 0 && e.mode == EPI_FWD && e.bias != nullptr && lane < 2 && (!TAIL || n0 < p.valid_n))
        prefetch_l1(e.bias + n0 + lane * 32);
      const long long e0 = (p.dbg && ew == 0 && lane == 0) ? clock64() : 0;
      mbar_wait(tfull_bar(st_, acc), acc_phase);
      tc_fence_after();
      if (p.dbg_flags & 1) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(st_, acc));
        continue;
      }
      if (p.dbg && ew == 0 && lane == 0) p.dbg[(size_t)blockIdx.x * 8 + 5] += clock64() - e0;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc_col(st_, acc) + (uint32_t)(half * kColW);
      if constexpr (NSLAB == 0) {
        // fp32 split-K partials straight from registers: this warp owns 32 rows x BN/2 columns, drained 32 columns at a time
        const bool do_bias = want_dbias && nblk == 0 && half == 0;
        float* o = (float*)e.out + (size_t)split * p.M * e.ldc + (size_t)grow * e.ldc + n0;
#pragma unroll
        for (int c = 0; c < BN / 64; ++c) {
          uint32_t raw[32];
          tc_ld32(taddr + 32u * c, raw);
          tc_wait_ld();
          if (grow < p.M) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (n0 + 32 * c + 4 * j + 3 < p.valid_n)
                reinterpret_cast<float4*>(o + 32 * c)[j] = make_float4(__uint_as_float(raw[4 * j]), __uint_as_float(raw[4 * j + 1]),
                                                                       __uint_as_float(raw[4 * j + 2]), __uint_as_float(raw[4 * j + 3]));
          }
        }
        if (do_bias) {
          uint32_t rawb[16];
          tc_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + bias_col(st_, acc), rawb);
          tc_wait_ld();
          if (grow < p.M) p.dbias_part[(size_t)split * p.M + grow] = __uint_as_float(rawb[0]);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(st_, acc));
        continue;
      }
      uint32_t raw0[32], raw1[32];
      tc_ld32(taddr, raw0);
      tc_ld32(taddr + 32u, raw1);
      tc_wait_ld();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {  // accumulator drained into registers: hand the TMEM stage back to the (leader's) MMA warp
        if (PAIR && !is_leader) mbar_arrive_remote(mapa_rank(tempty_bar(st_, acc), 0));
        else mbar_arrive(tempty_bar(st_, acc));
      }

      float v[64];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        v[j] = __uint_as_float(raw0[j]);
        v[32 + j] = __uint_as_float(raw1[j]);
      }
      if (stores_pending) {  // the previous tile's TMA stores must have finished reading the slabs
        if (lane == 0 && !p.has_in) tma_store_wait_read();  // (with an input operand lane 0 already waited before refilling the slab)
        __syncwarp();
      }
      if (e.mode == EPI_FWD) {
        if (e.bias != nullptr && (!TAIL || n0 < p.valid_n)) {
          const float4* b4 = reinterpret_cast<const float4*>(e.bias + n0);
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float4 b = __ldg(b4 + j);
            v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
          }
        }
        if (p.out3 && e.pos != nullptr && (!TAIL || n0 < p.valid_n)) {  // + pos_emb[token] (fp32), token of this thread's row
          const int tok = e.rm_offset + grow % e.rm_group;
          const float4* p4 = reinterpret_cast<const float4*>(e.pos + (size_t)tok * p.N + n0);
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float4 q = __ldg(p4 + j);
            v[4 * j] += q.x; v[4 * j + 1] += q.y; v[4 * j + 2] += q.z; v[4 * j + 3] += q.w;
          }
        }
        if (p.has_pre && NSLAB > 1) slab_store_row64(slab_pre, lane, v);
        if (p.has_pre && NSLAB == 1) {
          // ONE slab per warp (a second one would cost every stream a ring stage, and ring depth is what bounds these kernels):
          // the pre-activation goes out first through the same slab the output uses afterwards.  A prefetched residual lives in
          // that slab: it moves to registers (packed) before the slab is reused.
          uint32_t rp[32];
          if (p.has_in) {
            mbar_wait(in_bar(ew), in_phase);
            in_phase ^= 1u;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const uint32_t addr = slab_in + (uint32_t)lane * 128u + (uint32_t)((j ^ (lane & 7)) << 4);
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(rp[4 * j]), "=r"(rp[4 * j + 1]), "=r"(rp[4 * j + 2]), "=r"(rp[4 * j + 3]) : "r"(addr) : "memory");
            }
          }
          slab_store_row64(slab_out, lane, v);  // (a lane reads and writes only its own row)
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tma_pre, slab_out, n0, m0 + quarter * 32);
            tma_store_commit();
          }
          // the GELU arithmetic runs while the TMA engine reads the pre-activation out of the slab
          if (e.gelu) {
#pragma unroll
            for (int j = 0; j < 64; ++j) v[j] = gelu_bf16_f(v[j]);
          }
          if constexpr (DROP) { if (dropping) drop64(v, grow, n0); }
          if (p.has_in) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float2 r = unpack_bf16x2(rp[j]);
              v[2 * j] += r.x;
              v[2 * j + 1] += r.y;
            }
          }
          if (lane == 0) tma_store_wait_read();  // ... which must be done before the output is staged in the same slab
          __syncwarp();
        } else {
        if (e.gelu) {
#pragma unroll
          for (int j = 0; j < 64; ++j) v[j] = gelu_bf16_f(v[j]);
        }
        if constexpr (DROP) { if (dropping) drop64(v, grow, n0); }
        if (p.has_in) {
          mbar_wait(in_bar(ew), in_phase);
          in_phase ^= 1u;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float r[8];
            slab_load_chunk8(slab_in, lane, j, r);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[8 * j + i] += r[i];
          }
        }
        }
      } else {  // EPI_DGRAD
        if (p.has_in) {
          mbar_wait(in_bar(ew), in_phase);
          in_phase ^= 1u;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float z[8];
            slab_load_chunk8(slab_in, lane, j, z);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[8 * j + i] *= gelu_grad_bf16_f(z[i]);
          }
        }
        if constexpr (DROP) { if (dropping) drop64(v, grow, n0); }
      }
      slab_store_row64(slab_out, lane, v);
      fence_async_smem();  // generic-proxy smem writes -> visible to the TMA (async proxy)
      __syncwarp();
      if (lane == 0) {
        if (p.out3) {  // the slab's 32 rows are whole tokens of one image, or all tokens of 32 / rm_group consecutive images
          const int row0 = m0 + quarter * 32;
          tma_store_3d(&tma_out, slab_out, n0, e.rm_offset + row0 % e.rm_group, row0 / e.rm_group);  // images >= B are clipped
        } else {
          tma_store_2d(&tma_out, slab_out, n0, m0 + quarter * 32);  // rows >= M are clipped by the tensor map
        }
        if (p.has_pre && NSLAB > 1) tma_store_2d(&tma_pre, slab_pre, n0, m0 + quarter * 32);
        tma_store_commit();
      }
      stores_pending = true;
    }
    // the shared-memory source must have been read before the CTA exits; the global writes themselves complete with the grid
    // (what dependents wait for), so the kernel's tail does not sit out their round trip
    if (stores_pending && lane == 0) {
      if (kTailWaitRead) tma_store_wait_read();
      else tma_store_wait_all();
    }
  }

  // teardown: everyone (of both CTAs of a pair) done with TMEM and with remote barriers before the owning warp frees it
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();
  if (warp == NS) {
    tc_fence_after();
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}
