// shade2_body.cuh — the body of wf_shade2_kernel and wf_shade2_env_kernel (shade2.cuh), included inside both kernels.
// It is text, not a device function, because the compiler schedules a kernel that calls an inlined body differently
// from one that holds the code itself: so every shade kernel that existed before the environment map keeps its
// machine code. The including kernel provides kCount, kPerlinShared, kOrder, kAdaptive, kEnv and the parameters
// a, accum, active_out and counters.
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int i = blockIdx.x * blockDim.x + tid;
    const bool valid = i < a.n_slots;
    int32_t stack[kStackSize];  // only a ConstantMedium with a general boundary traverses here
    Tally<kCount> tally;

    int bounce = valid ? a.pool.bounce[i] : -2;
    const bool dry = __ldcg(a.next_item) >= a.total_items;  // read now, needed after the shading: its latency is covered
    if constexpr (kPerlinShared) {
        __shared__ DPerlin s_perlin;
        static_assert(sizeof(DPerlin) % 16 == 0, "DPerlin is copied in 16-byte words");
        const uint4* src = reinterpret_cast<const uint4*>(a.sc.perlins);
        uint4* dst = reinterpret_cast<uint4*>(&s_perlin);
        for (int k = tid; k < (int)(sizeof(DPerlin) / 16); k += kShadeBlock) dst[k] = __ldg(src + k);
        __syncthreads();
        a.sc.perlins = &s_perlin;
    }

    // ---- shade: media first (a scatter point in front of the surface hit replaces it), then one level of color() ----
    RayD ray{mk(0, 0, 0), mk(0, 0, 1), 0.0};
    PathColor pc{1.f, 1.f, 1.f, 0.f, 0.f, 0.f};
    Sampler smp{a.k0, a.k1, 0u, 0u, 0u};
    bool fresh = false;
    int32_t src_rec = -1;  // the record the new ray starts on (kOrder)
    if (bounce >= 0) {
        ray.o = mk(a.pool.ox[i], a.pool.oy[i], a.pool.oz[i]);
        ray.d = mk(a.pool.dx[i], a.pool.dy[i], a.pool.dz[i]);
        ray.time = a.pool.time[i];
        Best best{a.pool.best_t[i], a.pool.best_rec[i], a.pool.best_chain[i]};
        pc = PathColor{a.pool.thr_r[i], a.pool.thr_g[i], a.pool.thr_b[i], 0.f, 0.f, 0.f};
        smp.pixel = a.pool.pixel[i];
        smp.sample = a.pool.sample[i];
        smp.bounce = (uint32_t)bounce;
        if (a.sc.n_media > 0) media_after(a.sc, ray, 0.001, best, smp, stack, tally);
        bool ended;
        if (kEnv && best.rec < 0) {  // Q8 with the environment: the path ends like shade_hit's background branch
            const float3 e = env_lookup(a.env, ray.d);
            pc.rad_r += pc.thr_r * e.x; pc.rad_g += pc.thr_g * e.y; pc.rad_b += pc.thr_b * e.z;
            ended = true;
        } else {
            Albedo al;
            ended = shade_hit<false, kPerlinShared>(a.sc, a.cam.background, a.max_depth, ray, best, smp, pc, bounce, al);
            apply_albedo(pc, al);
        }
        if (ended) {
            atomicAdd(accum + smp.pixel, make_float4(pc.rad_r, pc.rad_g, pc.rad_b, 1.0f));  // one path sample done
            if constexpr (kAdaptive)
                if (smp.sample & 1u) atomicAdd(a.adaptive.aux + smp.pixel, make_float4(pc.rad_r, pc.rad_g, pc.rad_b, 1.0f));
            bounce = -1;
            a.pool.bounce[i] = -1;
        } else {
            fresh = true;
            src_rec = best.rec;
        }
    }
    {   // ---- refill empty slots per warp: consecutive items are the 32 pixels of one 8x4 tile at one sample index ----
        const bool want = bounce == -1;
        unsigned m = dry ? 0u : __ballot_sync(FULL, want);
        if (m != 0) {
            const int leader = __ffs(m) - 1;
            unsigned long long base = 0;
            if (lane == leader) base = atomicAdd(a.next_item, (unsigned long long)__popc(m));
            base = __shfl_sync(FULL, base, leader);
            const unsigned long long item = base + (unsigned long long)__popc(m & ((1u << lane) - 1u));
            if (want && item < a.total_items) {
                const unsigned long long group = item >> 5;
                const unsigned int tile = (unsigned int)(group / (unsigned long long)a.spp_count);
                const unsigned int smp_i = (unsigned int)(group - (unsigned long long)tile * (unsigned long long)a.spp_count);
                int tx, ty;
                tile_of_order(kAdaptive ? __ldg(a.adaptive.tile_list + tile) : tile, a.tiles_x, a.tiles_y, a.inv_per_block_row, tx, ty);
                const int pi = (int)(item & 31ull);
                const int px = tx * kTileW + (pi & (kTileW - 1));
                const int row = ty * kTileH + (pi / kTileW);  // row 0 = top
                if (px < a.width && row < a.height) {
                    smp.pixel = (uint32_t)(row * a.width + px);
                    smp.sample = (uint32_t)a.spp_begin + smp_i;
                    smp.bounce = 0;
                    camera_ray(a.cam, a.width, a.height, px, a.height - 1 - row, smp, ray);
                    pc = PathColor{1.f, 1.f, 1.f, 0.f, 0.f, 0.f};
                    bounce = 0;
                    fresh = true;
                }
            }
        }
    }
    // ---- the new ray goes to the pool with nothing hit yet: the trace kernel searches [0.001, inf) ----
    if (fresh) {
        a.pool.ox[i] = ray.o.x; a.pool.oy[i] = ray.o.y; a.pool.oz[i] = ray.o.z;
        a.pool.dx[i] = ray.d.x; a.pool.dy[i] = ray.d.y; a.pool.dz[i] = ray.d.z;
        a.pool.time[i] = ray.time;
        a.pool.best_t[i] = 1.7976931348623157e308; a.pool.best_rec[i] = -1; a.pool.best_chain[i] = 0;
        a.pool.thr_r[i] = pc.thr_r; a.pool.thr_g[i] = pc.thr_g; a.pool.thr_b[i] = pc.thr_b;
        a.pool.pixel[i] = smp.pixel; a.pool.sample[i] = smp.sample;
        a.pool.bounce[i] = bounce;
    }
    if constexpr (kOrder) {  // this slot's place in the next trace pass (order.cuh)
        uint2 kr = make_uint2(kOrderDead, 0u);
        if (fresh) kr.x = order_key(a.order, src_rec, ray.d.x, ray.d.y, ray.d.z);
        {   // one atomic per distinct key of the warp (camera rays of a refill share theirs: 32 same-address atomics
            // per warp cost the shade pass +50 us on every scene when each lane did its own)
            const unsigned same = __match_any_sync(FULL, kr.x);
            const int leader = __ffs(same) - 1;
            uint32_t base = 0;
            if (fresh && lane == leader) base = atomicAdd(a.order.hist + kr.x, (uint32_t)__popc(same));
            base = __shfl_sync(FULL, base, leader);
            kr.y = base + (uint32_t)__popc(same & ((1u << lane) - 1u));
        }
        if (valid) a.order.key_rank[i] = kr;
        order_scan_by_last_cta<kShadeBlock>(a.order, tid);
    }
    if (active_out) {
        const unsigned am = __ballot_sync(FULL, fresh);
        if (lane == 0 && am != 0) atomicAdd(active_out, (unsigned int)__popc(am));
    }
    if constexpr (kCount) {
        uint32_t v = tally.n_med;
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(FULL, v, off);
        if (lane == 0 && v) atomicAdd(&counters->medium_tests, (unsigned long long)v);
    }
