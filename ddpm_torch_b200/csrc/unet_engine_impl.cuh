// UNet engine, part 2: block builders (forward ops + adjoint tape), batched attention matmuls, plan().
#pragma once
#include <cmath>
#include "unet_engine.cuh"

namespace ddpm {

// the narrow convolutions' per-channel-count kernels (image channels 1..16)
inline void launch_im2col3(int ci, int nblk, cudaStream_t st, const float* src, bf16* dst, int B, int H, int W, int sign, const QsamplePro& qp) {
    switch (ci) {
        case 1: launch_k(k_im2col3<1>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 2: launch_k(k_im2col3<2>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 3: launch_k(k_im2col3<3>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 4: launch_k(k_im2col3<4>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 5: launch_k(k_im2col3<5>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 6: launch_k(k_im2col3<6>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 7: launch_k(k_im2col3<7>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 8: launch_k(k_im2col3<8>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 9: launch_k(k_im2col3<9>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 10: launch_k(k_im2col3<10>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 11: launch_k(k_im2col3<11>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 12: launch_k(k_im2col3<12>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 13: launch_k(k_im2col3<13>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 14: launch_k(k_im2col3<14>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        case 15: launch_k(k_im2col3<15>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
        default: launch_k(k_im2col3<16>, nblk, 256, 0, st, src, dst, B, H, W, sign, qp); break;
    }
}
// (out_conv with 4 channels takes the CUDA-core k_out_conv<4>: 36 tap outputs do not fit the 32-wide route)
inline void launch_out_gather(int co, int nblk, cudaStream_t st, const float* T, const float* bias, float* out, int B, int H, int W, const PsampleEpi& ps) {
    switch (co) {
        case 1: launch_k(k_out_gather<1>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 2: launch_k(k_out_gather<2>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 3: launch_k(k_out_gather<3>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 5: launch_k(k_out_gather<5>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 6: launch_k(k_out_gather<6>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 7: launch_k(k_out_gather<7>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 8: launch_k(k_out_gather<8>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 9: launch_k(k_out_gather<9>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 10: launch_k(k_out_gather<10>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 11: launch_k(k_out_gather<11>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 12: launch_k(k_out_gather<12>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 13: launch_k(k_out_gather<13>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 14: launch_k(k_out_gather<14>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        case 15: launch_k(k_out_gather<15>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
        default: launch_k(k_out_gather<16>, nblk, 256, 0, st, T, bias, out, B, H, W, ps); break;
    }
}

// Batched matmuls of the attention block (unet.py:43-51) and their adjoints.
//   form 0 (NT): C[b][i][j] = alpha * sum_c A[b][i][c] * B[b][j][c]     M=i, N=j, K=c
//   form 1 (NN): C[b][i][c] = sum_j A[b][i][j] * B[b][j][c]             M=i, N=c, K=j
//   form 2 (TN): C[b][j][c] = sum_i A[b][i][j] * B[b][i][c]             M=j, N=c, K=i
// A, B bf16 with row strides lda/ldb and per-batch strides = rows*ld; C bf16 or fp32.
inline void UnetEngine::bmm(std::vector<Op>& L, const std::string& name, int form, const bf16* A, long long lda, long long sa,
                            const bf16* Bp, long long ldb, long long sb, void* C, long long ldc, long long sc, bool c_f32,
                            int nb, int T, int Cc, float alpha, double* fl_acc) {
    // all attention products here are T x T x Cc shaped
    const int M = T, N = (form == 0) ? T : Cc, K = (form == 0) ? Cc : T;
    const double fl = 2.0 * nb * (double)M * N * K;
    if (fl_acc) *fl_acc += fl;
    const bool tc = (T % 128 == 0) && (Cc % 64 == 0) && ((T & (T - 1)) == 0);
    if (tc) {
        ddpm_gemm_desc d; memset(&d, 0, sizeof d);
        d.M = M; d.N = N; d.W = T; d.H = 1; d.NB = nb; d.alpha = alpha; d.grid_z = nb;
        d.out = C; d.ldo = (int)ldc; d.out_z_stride = sc; d.flags = c_f32 ? EPI_OUT_F32 : 0;
        d.a_ptr[0] = A; d.a_ld[0] = lda;
        if (form == 0) {
            d.mode = GEMM_KK; d.a_C[0] = K; d.nseg = 1; d.seg_map[0] = 0; d.seg_taps[0] = 1; d.seg_kchunks[0] = K / 64; d.seg_cbase[0] = 0;
            d.b_ptr = Bp; d.b_K = K; d.b_rows = N; d.b_batch = nb; d.b_ld = ldb; d.b_bs = sb; d.a_z_n = 1; d.b_z = 1;
        } else if (form == 1) {
            d.mode = GEMM_KMN; d.a_C[0] = K; d.b_ptr = Bp; d.b_K = N; d.b_ld = ldb; d.kblocks = K / 64; d.a_z_n = 1;
        } else {
            d.mode = GEMM_MNMN; d.a_C[0] = M; d.b_ptr = Bp; d.b_K = N; d.b_ld = ldb; d.taps = 1; d.splits = 1; d.kblocks = K / 64;
        }
        ++n_tc_gemms;
        if (dry) { push(L, name, fl, [](cudaStream_t) { return 0; }); return; }
        GemmLaunch g; int rc = build_gemm(d, g);
        if (rc) { plan_error = rc; return; }
        push(L, name, fl, [g](cudaStream_t st) { return launch_gemm(g, st); });
        return;
    }
    ++n_generic;
    SgemmParams p; memset(&p, 0, sizeof p);
    p.A = A; p.B = Bp; p.C = C; p.M = M; p.N = N; p.K = K; p.alpha = alpha;
    p.sa_z = sa; p.sb_z = sb; p.sc_z = sc; p.sc_m = ldc; p.sc_n = 1;
    if (form == 0) { p.sa_m = lda; p.sa_k = 1; p.sb_k = 1; p.sb_n = ldb; }
    else if (form == 1) { p.sa_m = lda; p.sa_k = 1; p.sb_k = ldb; p.sb_n = 1; }
    else { p.sa_m = 1; p.sa_k = lda; p.sb_k = ldb; p.sb_n = 1; }
    const dim3 grid((N + 63) / 64, (M + 63) / 64, nb);
    if (c_f32) push(L, name + "[simt]", fl, [p, grid](cudaStream_t st) { launch_k(k_sgemm<bf16, bf16, float>, grid, 256, 0, st, p); return (int)cudaGetLastError(); });
    else       push(L, name + "[simt]", fl, [p, grid](cudaStream_t st) { launch_k(k_sgemm<bf16, bf16, bf16>, grid, 256, 0, st, p); return (int)cudaGetLastError(); });
}

// ResidualBlock (unet.py:63-89):  out = skip(x) + conv2(drop(silu(gn2(conv1(silu(gn1(x))) + fc(silu(temb))))))
inline T4 UnetEngine::res_block(const std::string& p, const Src& x, int cout, int tp_off, int tp_ld, float* TP, float* dTP) {
    const int cin = x.C(), Bn = x.t0.B, h = x.t0.H, w = x.t0.W;
    const bool has_skip = cin != cout;
    // inference plans: norm + SiLU ride in the consumer conv's operand path (no `a` tensor, no apply pass) where the conv can
    const bool xf1 = xf_ok(x, cout, h, w);
    T4 a1; GnSaved g1{}; const float* K1 = nullptr;
    if (xf1) K1 = gn_prep_xf(fwd_ops, p + ".norm1", x, p + ".norm1");
    else { a1 = newT(Bn, h, w, cin); g1 = gn_fwd(fwd_ops, p + ".norm1", x, p + ".norm1", a1, 1, 0.f); }
    const Packed w1 = pack_conv(p + ".conv1", cout, cin, 3, 0, true, true);
    T4 h1 = newT(Bn, h, w, cout);
    {
        ConvSpec c; c.name = p + ".conv1"; c.in = xf1 ? x : one(a1); c.xfK = K1; c.xf_silu = 1; c.wp = w1.fwd; c.ldw = w1.ld_f; c.bias = PP(p + ".conv1.bias");
        c.rowvec = TP + tp_off; c.rowvec_ld = tp_ld; c.out = h1; c.Co = cout; c.Ho = h; c.Wo = w;
        c.want_qstats = true;                       // h1 feeds norm2: its statistics come out of this conv's epilogue
        h1.qs = conv_op(fwd_ops, c, &fwd_flops);
    }
    const bool xf2 = xf_ok(one(h1), cout, h, w);
    T4 a2; GnSaved g2{}; const float* K2 = nullptr;
    if (xf2) K2 = gn_prep_xf(fwd_ops, p + ".norm2", one(h1), p + ".norm2");
    else { a2 = newT(Bn, h, w, cout); g2 = gn_fwd(fwd_ops, p + ".norm2", one(h1), p + ".norm2", a2, 1, cfg.drop_rate); }
    // identity residual (cin == cout) of a conv that takes the haloed kernel: x rides in as two extra K chunks with identity weights
    // (exact: 1.0 * bf16 accumulated in fp32) instead of a 64-byte-per-lane global read in the epilogue, which made these convs
    // epilogue-bound (bs=256, 128->128 at 32x32: 90 us against 66 us for the same conv without residual).  Three convs of the CIFAR
    // net qualify: sampler step 4.303 -> 4.291 ms, training step 9.127 -> 9.111 ms (A/B via DDPM_NO_IDENTITY_SKIP)
    static const bool no_idskip = getenv("DDPM_NO_IDENTITY_SKIP") != nullptr;
    const bool id_skip = !has_skip && !no_idskip && !x.two && cout % 64 == 0 && halo_eligible(h, w, cout) && tc_ok_geom(h, w) && !getenv("DDPM_NO_HALO");
    const Packed w2 = pack_conv(p + ".conv2", cout, cout, 3, has_skip ? cin : (id_skip ? cout : 0), true, true);
    if (id_skip) pack_identity(w2, 9 * cout, cout);
    bf16* wsd = nullptr; float* bias2 = PP(p + ".conv2.bias");
    if (has_skip) {
        if (train) wsd = at<bf16>(alloc((size_t)cin * cout * 2));
        pack_extra(p + ".skip", w2, 9 * cout, cout, cin, wsd, cout);
        float* comb = at<float>(alloc((size_t)cout * 4));
        pack_bias_add(comb, PP(p + ".conv2.bias"), PP(p + ".skip.bias"), cout);
        bias2 = comb;
    }
    T4 out = newT(Bn, h, w, cout);
    {
        ConvSpec c; c.name = p + ".conv2"; c.in = xf2 ? one(h1) : one(a2); c.xfK = K2; c.xf_silu = 1; c.wp = w2.fwd; c.ldw = w2.ld_f; c.bias = bias2;
        c.has_skip = has_skip || id_skip; c.skip_identity = id_skip; c.skip_in = x; c.residual = (has_skip || id_skip) ? nullptr : bp(x.t0);
        c.out = out; c.Co = cout; c.Ho = h; c.Wo = w;
        c.want_qstats = true;                       // block outputs feed the next norm1 / attention norm / out_conv.0 (and, as skips, the up path)
        out.qs = conv_op(fwd_ops, c, &fwd_flops);
    }
    if (!train) return out;
    tape_push([=]() {
        const T4 dOut = grad_of(out, nullptr);
        colsum_op(p + ".conv2.bias", dOut, nullptr, 0, GP(p + ".conv2.bias"), has_skip ? GP(p + ".skip.bias") : nullptr, cout);
        T4 d_a2 = newT(Bn, h, w, cout);
        { ConvSpec c; c.name = p + ".conv2.dgrad"; c.in = one(dOut); c.wp = w2.dgr; c.ldw = w2.ld_d; c.out = d_a2; c.Co = cout; c.Ho = h; c.Wo = w;
          conv_op(bwd_ops, c, &bwd_flops); }
        wgrad_op(p + ".conv2.wgrad", dOut, one(a2), 3, 1, MAP_NORMAL, GP(p + ".conv2.weight"), cout);
        T4 dxs;
        if (has_skip) {
            dxs = newT(Bn, h, w, cin);
            ConvSpec c; c.name = p + ".skip.dgrad"; c.in = one(dOut); c.ksize = 1; c.wp = wsd; c.ldw = cout; c.out = dxs; c.Co = cin; c.Ho = h; c.Wo = w;
            conv_op(bwd_ops, c, &bwd_flops);
            wgrad_op(p + ".skip.wgrad", dOut, x, 1, 1, MAP_NORMAL, GP(p + ".skip.weight"), cout);
        }
        // the column sums of d_h1 (bias gradients of conv1 / fc and the per-image timestep-projection gradient) are
        // accumulated by the same kernel that produces d_h1
        gn_bwd(p + ".norm2", g2, d_a2, nullptr, dTP + tp_off, tp_ld, GP(p + ".conv1.bias"), GP(p + ".fc.bias"));
        const T4 d_h1 = grad_of(h1, nullptr);
        T4 d_a1 = newT(Bn, h, w, cin);
        { ConvSpec c; c.name = p + ".conv1.dgrad"; c.in = one(d_h1); c.wp = w1.dgr; c.ldw = w1.ld_d; c.out = d_a1; c.Co = cin; c.Ho = h; c.Wo = w;
          conv_op(bwd_ops, c, &bwd_flops); }
        wgrad_op(p + ".conv1.wgrad", d_h1, one(a1), 3, 1, MAP_NORMAL, GP(p + ".conv1.weight"), cout);
        gn_bwd(p + ".norm1", g1, d_a1, has_skip ? bp(dxs) : bp(dOut));
    });
    return out;
}

// AttentionBlock (unet.py:23-60): out = x + Wo . softmax(Q^T K / sqrt(C)) V ,  q,k,v = chunk(Win . gn(x))
inline T4 UnetEngine::attn_block(const std::string& p, const T4& x) {
    const int C = x.C, Bn = x.B, h = x.H, w = x.W, T = h * w;
    const float scale = 1.f / sqrtf((float)C);
    T4 xn = newT(Bn, h, w, C);
    const GnSaved g = gn_fwd(fwd_ops, p + ".norm", one(x), p + ".norm", xn, 0, 0.f);
    const Packed win = pack_conv(p + ".project_in", 3 * C, C, 1, 0, false, true);
    T4 qkv = newT(Bn, h, w, 3 * C);
    { ConvSpec c; c.name = p + ".project_in"; c.in = one(xn); c.ksize = 1; c.wp = win.fwd; c.ldw = win.ld_f; c.bias = PP(p + ".project_in.bias");
      c.out = qkv; c.Co = 3 * C; c.Ho = h; c.Wo = w; conv_op(fwd_ops, c, &fwd_flops); }
    const bf16* q = bp(qkv);
    const long long ldq = 3 * C, sq = (long long)T * 3 * C;
    T4 O = newT(Bn, h, w, C);
    float* S = nullptr; bf16* Pm = nullptr;
    static const bool no_fused_attn = getenv("DDPM_NO_FUSED_ATTN") != nullptr;
    static const bool no_attn16 = getenv("DDPM_NO_ATTN16") != nullptr;
    const bool small16 = !no_attn16 && attn16_eligible(T, C);
    // OPT-IN (DDPM_FUSED_ATTN_BWD=1, read at plan time): dP -> softmax backward -> dQ as one launch is parity-green and 3x shorter than
    // the three launches it replaces, but its 214 KB CTAs cannot co-reside with the weight-gradient GEMMs of the side stream
    // and the whole step is 0.3 % slower (9.21 vs 9.18 ms); profiles/r02_attention_backward_experiment.txt
    const bool fused_attn_bwd = getenv("DDPM_FUSED_ATTN_BWD") != nullptr;
    const bool fused_bwd = train && fused_attn_bwd && !no_fused_attn && attn_fused_eligible(T, C);
    static const bool no_fused_attn_train = getenv("DDPM_NO_FUSED_ATTN_TRAIN") != nullptr;
    if (!(train && no_fused_attn_train) && !no_fused_attn && attn_fused_eligible(T, C)) {
        // Q.K^T -> softmax -> P.V in ONE kernel, S and O in TMEM, P in shared memory (attn_fused.cuh); training plans also get
        // the normalised P in HBM for the backward pass
        if (train) Pm = at<bf16>(alloc((size_t)Bn * T * T * 2));
        const double fl = 4.0 * Bn * (double)T * T * C;
        fwd_flops += fl; ++n_tc_gemms;
        if (dry) push(fwd_ops, p + ".attn[fused]", fl, [](cudaStream_t) { return 0; });
        else {
            AttnLaunch g; const int rc = build_attn(q, bp(O), Bn, T, C, g, Pm);
            if (rc) { plan_error = rc; return O; }
            push(fwd_ops, p + ".attn[fused]", fl, [g](cudaStream_t st) { return launch_attn(g, st); });
        }
    } else if (small16) {
        // 4x4 level: one CTA per image does scores, softmax and P.V (k_attn16_fwd); P is kept only when a backward follows
        if (train) Pm = at<bf16>(alloc((size_t)Bn * T * T * 2));
        const double fl = 4.0 * Bn * (double)T * T * C;
        fwd_flops += fl; ++n_generic;
        bf16* Op = bp(O); bf16* Pk = Pm; const size_t shm = attn16_smem(C, false);
        if (!dry) cudaFuncSetAttribute(k_attn16_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn16_smem(512, false));
        push(fwd_ops, p + ".attn[t16]", fl, [=](cudaStream_t st) { launch_k(k_attn16_fwd, Bn, 256, shm, st, q, Op, Pk, C, scale); return (int)cudaGetLastError(); });
    } else {
        S = at<float>(alloc((size_t)Bn * T * T * 4));
        Pm = at<bf16>(alloc((size_t)Bn * T * T * 2));
        bmm(fwd_ops, p + ".qk", 0, q, ldq, sq, q + C, ldq, sq, S, T, (long long)T * T, true, Bn, T, C, scale, &fwd_flops);
        { const long long rows = (long long)Bn * T; const int nblk = (int)((rows + 7) / 8);
          push(fwd_ops, p + ".softmax", 0, [=](cudaStream_t st) { launch_k(k_softmax_rows, nblk, 256, 0, st, S, Pm, rows, T); return (int)cudaGetLastError(); }); }
        bmm(fwd_ops, p + ".pv", 1, Pm, T, (long long)T * T, q + 2 * C, ldq, sq, bp(O), C, (long long)T * C, false, Bn, T, C, 1.f, &fwd_flops);
    }
    const Packed wout = pack_conv(p + ".project_out", C, C, 1, 0, false, true);
    T4 out = newT(Bn, h, w, C);
    { ConvSpec c; c.name = p + ".project_out"; c.in = one(O); c.ksize = 1; c.wp = wout.fwd; c.ldw = wout.ld_f; c.bias = PP(p + ".project_out.bias");
      c.residual = bp(x); c.out = out; c.Co = C; c.Ho = h; c.Wo = w; c.want_qstats = true; out.qs = conv_op(fwd_ops, c, &fwd_flops); }
    if (!train) return out;
    tape_push([=]() {
        const T4 dY = grad_of(out, nullptr);
        colsum_op(p + ".project_out.bias", dY, nullptr, 0, GP(p + ".project_out.bias"), nullptr, C);
        T4 dO = newT(Bn, h, w, C);
        { ConvSpec c; c.name = p + ".project_out.dgrad"; c.in = one(dY); c.ksize = 1; c.wp = wout.dgr; c.ldw = wout.ld_d; c.out = dO; c.Co = C; c.Ho = h; c.Wo = w;
          conv_op(bwd_ops, c, &bwd_flops); }
        wgrad_op(p + ".project_out.wgrad", dY, one(O), 1, 1, MAP_NORMAL, GP(p + ".project_out.weight"), C);
        T4 dqkv = newT(Bn, h, w, 3 * C);
        const bf16* dOp = bp(dO); bf16* dq = bp(dqkv);
        if (small16) {
            const double fl = 8.0 * Bn * (double)T * T * C;
            bwd_flops += fl; ++n_generic;
            const size_t shm = attn16_smem(C, true); const bf16* Pk = Pm;
            if (!dry) cudaFuncSetAttribute(k_attn16_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn16_smem(512, true));
            push(bwd_ops, p + ".attn_bwd[t16]", fl, [=](cudaStream_t st) { launch_k(k_attn16_bwd, Bn, 256, shm, st, q, dOp, Pk, dq, C, scale); return (int)cudaGetLastError(); });
        } else if (fused_bwd) {
            // dP -> softmax backward -> dQ in one launch (attn_kernel<true>); dK and dV read dS / P back as GEMM operands
            bf16* dS = at<bf16>(alloc((size_t)Bn * T * T * 2));
            const double fl = 4.0 * Bn * (double)T * T * C;
            bwd_flops += fl; ++n_tc_gemms;
            if (dry) push(bwd_ops, p + ".attn_bwd[fused]", fl, [](cudaStream_t) { return 0; });
            else {
                AttnLaunch g; const int rc = build_attn_bwd(q, dOp, Pm, dS, dq, Bn, T, C, g);
                if (rc) { plan_error = rc; return; }
                push(bwd_ops, p + ".attn_bwd[fused]", fl, [g](cudaStream_t st) { return launch_attn_bwd(g, st); });
            }
            bmm(bwd_ops, p + ".dV", 2, Pm, T, (long long)T * T, dOp, C, (long long)T * C, dq + 2 * C, ldq, sq, false, Bn, T, C, 1.f, &bwd_flops);
            bmm(bwd_ops, p + ".dK", 2, dS, T, (long long)T * T, q, ldq, sq, dq + C, ldq, sq, false, Bn, T, C, 1.f, &bwd_flops);
        } else {
        float* dP = at<float>(alloc((size_t)Bn * T * T * 4));
        bf16* dS = at<bf16>(alloc((size_t)Bn * T * T * 2));
        bmm(bwd_ops, p + ".dP", 0, dOp, C, (long long)T * C, q + 2 * C, ldq, sq, dP, T, (long long)T * T, true, Bn, T, C, 1.f, &bwd_flops);
        bmm(bwd_ops, p + ".dV", 2, Pm, T, (long long)T * T, dOp, C, (long long)T * C, dq + 2 * C, ldq, sq, false, Bn, T, C, 1.f, &bwd_flops);
        { const long long rows = (long long)Bn * T; const int nblk = (int)((rows + 7) / 8);
          push(bwd_ops, p + ".softmax_bwd", 0, [=](cudaStream_t st) { launch_k(k_softmax_bwd, nblk, 256, 0, st, Pm, dP, dS, rows, T, scale); return (int)cudaGetLastError(); }); }
        bmm(bwd_ops, p + ".dQ", 1, dS, T, (long long)T * T, q + C, ldq, sq, dq, ldq, sq, false, Bn, T, C, 1.f, &bwd_flops);
        bmm(bwd_ops, p + ".dK", 2, dS, T, (long long)T * T, q, ldq, sq, dq + C, ldq, sq, false, Bn, T, C, 1.f, &bwd_flops);
        }
        colsum_op(p + ".project_in.bias", dqkv, nullptr, 0, GP(p + ".project_in.bias"), nullptr, 3 * C);
        T4 dxn = newT(Bn, h, w, C);
        { ConvSpec c; c.name = p + ".project_in.dgrad"; c.in = one(dqkv); c.ksize = 1; c.wp = win.dgr; c.ldw = win.ld_d; c.out = dxn; c.Co = C; c.Ho = h; c.Wo = w;
          conv_op(bwd_ops, c, &bwd_flops); }
        wgrad_op(p + ".project_in.wgrad", dqkv, one(xn), 1, 1, MAP_NORMAL, GP(p + ".project_in.weight"), 3 * C);
        gn_bwd(p + ".norm", g, dxn, bp(dY));
    });
    return out;
}

// Downsample (unet.py:163-167): SamePad2d(3,2) = zero-pad bottom/right by one, then 3x3 stride 2.
// Tensor-core path: forward / wgrad read the input through tensor maps with elementStrides 2; the data gradient is four
// output-parity sub-convolutions over dY (4+2+2+1 taps) whose epilogues scatter to the (2y+py, 2x+px) pixels.
inline T4 UnetEngine::down_conv(const std::string& p, const T4& x) {
    const int C = x.C, Bn = x.B, h = x.H, w = x.W;
    const bool tc = (C % 64 == 0) && tc_ok_geom(h / 2, w / 2);
    const Packed pk = pack_conv(p, C, C, 3, 0, /*flip=*/false, true, tc ? 3 : 1);
    T4 out = newT(Bn, h / 2, w / 2, C);
    { ConvSpec c; c.name = p; c.in = one(x); c.stride = 2; c.wp = pk.fwd; c.ldw = pk.ld_f; c.bias = PP(p + ".bias"); c.out = out; c.Co = C; c.Ho = h / 2; c.Wo = w / 2;
      c.want_qstats = true; out.qs = conv_op(fwd_ops, c, &fwd_flops); }
    if (!train) return out;
    tape_push([=]() {
        const T4 dY = grad_of(out, nullptr);
        colsum_op(p + ".bias", dY, nullptr, 0, GP(p + ".bias"), nullptr, C);
        bool first = true; const T4 dx = grad_of(x, &first);
        if (tc) {
            const double fl = 2.0 * dY.pix() * C * 9.0 * C;
            bwd_flops += fl;
            int q = 0;
            for (int py = 0; py < 2; ++py) for (int px = 0; px < 2; ++px, ++q) {
                ddpm_gemm_desc d; memset(&d, 0, sizeof d);
                d.mode = GEMM_KK; d.M = (int)dY.pix(); d.N = C; d.W = w / 2; d.H = h / 2; d.NB = Bn;
                d.a_ptr[0] = bp(dY); d.a_C[0] = C; d.a_ld[0] = C;
                d.nseg = 1; d.seg_map[0] = 0; d.seg_kchunks[0] = C / 64; d.seg_cbase[0] = 0; d.seg_custom[0] = 1; d.seg_cmul[0] = 1;
                int nt = 0;
                for (int ky = py ? 1 : 0; ky < 3; ky += 2) for (int kx = px ? 1 : 0; kx < 3; kx += 2) {
                    d.seg_dy[0][nt] = (signed char)(-(ky / 2)); d.seg_dx[0][nt] = (signed char)(-(kx / 2)); ++nt;
                    if (px) break;
                }
                // (the loops above enumerate ky in {0,2} or {1} and kx in {0,2} or {1}, kx fastest)
                d.seg_taps[0] = nt;
                d.b_ptr = pk.dgr; d.b_K = 9 * C; d.b_rows = C; d.b_batch = 1; d.b_ld = pk.ld_d;
                d.b_k_base = (py == 0 ? (px == 0 ? 0 : 4) : (px == 0 ? 6 : 8)) * C;
                d.out = bp(dx); d.ldo = C; d.alpha = 1.f; d.grid_z = 1; d.o_mul = 2; d.o_py = py; d.o_px = px;
                if (!first) { d.residual = bp(dx); d.ldr = C; }
                ++n_tc_gemms;
                if (dry) { push(bwd_ops, p + ".dgrad", q ? 0 : fl, [](cudaStream_t) { return 0; }); continue; }
                GemmLaunch g; const int rc = build_gemm(d, g);
                if (rc) { plan_error = rc; return; }
                push(bwd_ops, p + ".dgrad", q ? 0 : fl, [g](cudaStream_t st) { return launch_gemm(g, st); });
            }
        } else {
            ConvSpec c; c.name = p + ".dgrad"; c.in = one(dY); c.map = MAP_TRANSPOSED2; c.wp = pk.dgr; c.ldw = pk.ld_d; c.out = dx; c.Co = C; c.Ho = h; c.Wo = w; c.accumulate = !first;
            conv_op(bwd_ops, c, &bwd_flops);
        }
        wgrad_op(p + ".wgrad", dY, one(x), 3, 2, MAP_NORMAL, GP(p + ".weight"), C);
    });
    return out;
}

// Upsample (unet.py:199-202): nearest x2 then 3x3 conv
inline T4 UnetEngine::up_conv(const std::string& p, const T4& x) {
    const int C = x.C, Bn = x.B, h = x.H, w = x.W;
    static const bool no_fold = getenv("DDPM_NO_UPFOLD") != nullptr;
    // (128-channel layers keep the explicit form: their folded GEMMs have 128-wide tiles, which the shared-memory operand
    // bandwidth caps at ~2/3 of the MMA rate, and the haloed kernel on the 2x grid wins - CelebA-HQ 256^2: 6.16 vs 6.26 ms/step)
    if (!train && !no_fold && C % 256 == 0 && tc_ok_geom(h, w)) {
        // Inference plans: the upsampled tensor is never materialised.  Four output-parity sub-convolutions with 2x2 taps over the
        // low-resolution input (merged weights, PK_UPFOLD) scatter to the (2y+py, 2x+px) pixels: 4/9 of the MACs, no 2x copy.
        // (Training keeps the explicit form: the weight gradient wants the upsampled tensor as its operand.)
        Packed pk; pk.ld_f = 16LL * C; pk.fwd = at<bf16>(alloc((size_t)C * pk.ld_f * 2));
        { PackEntry e; memset(&e, 0, sizeof e); e.kind = PK_UPFOLD; e.Co = C; e.Ci = C; e.taps = 9; e.w = PP(p + ".weight"); e.fwd = pk.fwd; e.ld_f = pk.ld_f;
          pack_table_host.push_back(e); }
        T4 out = newT(Bn, 2 * h, 2 * w, C);
        const double fl = 2.0 * out.pix() * C * 9.0 * C;       // the reference's count (the folded form does 4/9 of it)
        fwd_flops += fl;
        ddpm_gn_epi gn; memset(&gn, 0, sizeof gn);
        static const bool no_fuse = getenv("DDPM_NO_GN_EPI") != nullptr;
        if (!no_fuse && C % 32 == 0 && (h * w) % 32 == 0) { out.qs = (long long)zero_fwd((size_t)Bn * (C / 4) * 2 * 8); gn.qstats = at<double>((size_t)out.qs); }
        for (int q = 0; q < 4; ++q) {
            const int py = q >> 1, px = q & 1;
            ddpm_gemm_desc d; memset(&d, 0, sizeof d);
            d.mode = GEMM_KK; d.M = (int)x.pix(); d.N = C; d.W = w; d.H = h; d.NB = Bn;
            d.a_ptr[0] = bp(x); d.a_C[0] = C; d.a_ld[0] = C;
            d.nseg = 1; d.seg_map[0] = 0; d.seg_kchunks[0] = C / 64; d.seg_cbase[0] = 0; d.seg_custom[0] = 1; d.seg_cmul[0] = 1; d.seg_taps[0] = 4;
            for (int a = 0; a < 2; ++a) for (int b = 0; b < 2; ++b) {
                d.seg_dy[0][a * 2 + b] = (signed char)(py == 0 ? a - 1 : a); d.seg_dx[0][a * 2 + b] = (signed char)(px == 0 ? b - 1 : b);
            }
            d.b_ptr = pk.fwd; d.b_K = 16 * C; d.b_rows = C; d.b_batch = 1; d.b_ld = pk.ld_f; d.b_k_base = q * 4 * C;
            d.out = bp(out); d.ldo = C; d.alpha = 1.f; d.grid_z = 1; d.o_mul = 2; d.o_py = py; d.o_px = px;
            d.bias = PP(p + ".bias"); d.gn = gn;
            ++n_tc_gemms;
            if (dry) { push(fwd_ops, p + "[fold]", q ? 0 : fl, [](cudaStream_t) { return 0; }); continue; }
            GemmLaunch g; const int rc = build_gemm(d, g);
            if (rc) { plan_error = rc; return out; }
            push(fwd_ops, p + "[fold]", q ? 0 : fl, [g](cudaStream_t st) { return launch_gemm(g, st); });
        }
        return out;
    }
    T4 up = newT(Bn, 2 * h, 2 * w, C);
    { const bf16* src = bp(x); bf16* dst = bp(up); const int n = grid_for((long long)Bn * 4 * h * w * (C / 8));
      push(fwd_ops, p + ".upsample", 0, [=](cudaStream_t st) { launch_k(k_upsample2x, n, 256, 0, st, src, dst, Bn, h, w, C); return (int)cudaGetLastError(); }); }
    const Packed pk = pack_conv(p, C, C, 3, 0, true, true);
    T4 out = newT(Bn, 2 * h, 2 * w, C);
    { ConvSpec c; c.name = p; c.in = one(up); c.wp = pk.fwd; c.ldw = pk.ld_f; c.bias = PP(p + ".bias"); c.out = out; c.Co = C; c.Ho = 2 * h; c.Wo = 2 * w;
      c.want_qstats = true; out.qs = conv_op(fwd_ops, c, &fwd_flops); }
    if (!train) return out;
    tape_push([=]() {
        const T4 dY = grad_of(out, nullptr);
        colsum_op(p + ".bias", dY, nullptr, 0, GP(p + ".bias"), nullptr, C);
        T4 dUp = newT(Bn, 2 * h, 2 * w, C);
        { ConvSpec c; c.name = p + ".dgrad"; c.in = one(dY); c.wp = pk.dgr; c.ldw = pk.ld_d; c.out = dUp; c.Co = C; c.Ho = 2 * h; c.Wo = 2 * w;
          conv_op(bwd_ops, c, &bwd_flops); }
        wgrad_op(p + ".wgrad", dY, one(up), 3, 1, MAP_NORMAL, GP(p + ".weight"), C);
        bool first = true; const T4 dx = grad_of(x, &first);
        const bf16* src = bp(dUp); bf16* dst = bp(dx); const int n = grid_for((long long)Bn * h * w * (C / 8)); const int acc = first ? 0 : 1;
        push(bwd_ops, p + ".upsample_bwd", 0, [=](cudaStream_t st) { launch_k(k_upsample2x_bwd, n, 256, 0, st, src, dst, Bn, h, w, C, acc); return (int)cudaGetLastError(); });
    });
    return out;
}

inline int UnetEngine::plan(int B_, int H_, int W_, bool train_, bool dry_) {
    B = B_; H = H_; W = W_; train = train_; dry = dry_;
    gemm_pair_hint() = train ? 0 : 1;               // CTA-pair GEMM kernels: inference plans only (measured, gemm_build.cuh)
    cursor = 0; pack_ops.clear(); fwd_ops.clear(); bwd_ops.clear(); tape.clear(); tape_tag.clear(); cur_tag = "late"; grads.clear(); once_list.clear();
    { std::vector<GradChunk> keep; keep.swap(chunks); for (auto& c : keep) if (c.ev) cudaEventDestroy(c.ev); }
    tp_table_host.clear(); tp_uni_table_host.clear(); fc_table_host.clear(); tpw_table_host.clear(); tpd_table_host.clear(); pack_table_host.clear(); unpack_table_host.clear();
    layer_counter = 0; fwd_flops = bwd_flops = 0; n_tc_gemms = n_generic = 0; plan_error = 0; gather_fused_tail = false;
    const size_t zf_total = zf_cursor, zb_total = zb_cursor;   // sizes learned by the preceding dry pass
    zf_cursor = zb_cursor = 0;
    zero_fwd_bytes = dry ? 0 : zf_total; zero_bwd_bytes = dry ? 0 : zb_total;
    zero_fwd_off = alloc(dry ? 0 : zf_total); zero_bwd_off = alloc(dry ? 0 : zb_total);
    const int ch = cfg.hid_channels, L = cfg.levels, nrb = cfg.num_res_blocks, E = cfg.temb_dim, Cin = cfg.in_channels, Cout = cfg.out_channels;
    if (ch % 32) return fail(-30, "hid_channels must be a multiple of 32 (GroupNorm(32))");
    if (Cin > 16 || Cin < 1 || Cout > 16 || Cout < 1) return fail(-30, "in_channels / out_channels must be 1..16 (image channels)");
    // 5..16 image channels (block-size models: C*b^2 channels at 1/b the resolution) exist only on the tensor-core routes of in_conv /
    // out_conv.2; the CUDA-core fallbacks stop at 4
    const bool wide_in = Cin > 4, wide_out = Cout > 4;
    if ((wide_in || wide_out) && !(ch % 64 == 0 && tc_ok_geom(H, W)))
        return fail(-30, "in_channels / out_channels of 5..16 need the tensor-core narrow convolutions: hid_channels %% 64 == 0 "
                         "and a tensor-core resolution (got hid_channels=%d, %dx%d)", ch, H, W);
    if ((H >> (L - 1)) < 1 || (H % (1 << (L - 1))) || (W % (1 << (L - 1)))) return fail(-30, "resolution not divisible by 2^(levels-1)");
    UnetEngine* self = this;

    // ---- diffusion-side buffers
    const size_t img_elems = (size_t)B * Cin * H * W;
    xt_off = alloc(img_elems * 4); eps_off = alloc((size_t)B * Cout * H * W * 4);
    tbuf_off = alloc((size_t)B * 8); coefcur_off = alloc(64); counter_off = alloc(64);
    deps_off = alloc((size_t)B * Cout * H * W * 4);

    // ---- zero the per-forward accumulators
    { uint8_t* z = ws + zero_fwd_off; const size_t n = zero_fwd_bytes;
      push(fwd_ops, "zero.fwd", 0, [z, n](cudaStream_t st) { return n ? (int)cudaMemsetAsync(z, 0, n, st) : 0; }, 0); }

    // ---- timestep embedding MLP (functions.py:10-26, unet.py:122-126) + all per-block projections (unet.py:77,86)
    int nblocks = L * nrb + 2 + L * (nrb + 1);
    int maxc = 0; for (int i = 0; i < L; ++i) if (chs(i) > maxc) maxc = chs(i);
    const int tp_ld = nblocks * maxc;
    float* emb = at<float>(alloc((size_t)B * ch * 4));
    float* e0 = at<float>(alloc((size_t)B * E * 4));
    float* e1 = at<float>(zero_fwd((size_t)B * E * 4));            // K-split GEMMs accumulate into zeroed outputs
    float* TP = at<float>(zero_fwd((size_t)B * tp_ld * 4));
    constexpr int KS = 4;
    float* dTP = at<float>(zero_bwd((size_t)B * tp_ld * 4));
    float* d_st = at<float>(zero_bwd((size_t)B * E * 4));
    tp_table_off = alloc(sizeof(SgemmParams) * nblocks); tpw_table_off = alloc(sizeof(SgemmParams) * nblocks); tpd_table_off = alloc(sizeof(SgemmParams) * nblocks);
    tp_uni_table_off = alloc(sizeof(SgemmParams) * nblocks);
    // tensor-core projections need a power-of-two batch (plain-matrix TMA boxes) and, for the weight gradient, B % 64 == 0
    static const bool no_tc_temb = getenv("DDPM_NO_TC_TEMB") != nullptr;
    const bool tc_temb = !no_tc_temb && (B & (B - 1)) == 0 && B >= 64 && E % 64 == 0 && maxc % 32 == 0 && tp_ld % 64 == 0;
    fc_table_off = alloc(sizeof(FcEnt) * nblocks);
    bf16* Wcat = tc_temb ? at<bf16>(alloc_once_zero((size_t)tp_ld * E * 2)) : nullptr;
    bf16* WcatT = (tc_temb && train) ? at<bf16>(alloc_once_zero((size_t)tp_ld * E * 2)) : nullptr;
    float* bias_cat = tc_temb ? at<float>(alloc_once_zero((size_t)tp_ld * 4)) : nullptr;
    bf16* A_f = tc_temb ? at<bf16>(alloc((size_t)B * E * 2)) : nullptr;
    const size_t temb_first = fwd_ops.size();
    {
        const int Bn = B;
        push(fwd_ops, "temb.sin", 0, [=](cudaStream_t st) { launch_k(k_timestep_embedding, (Bn * (ch / 2) + 127) / 128, 128, 0, st, self->t_in, emb, Bn, ch); return (int)cudaGetLastError(); });
        SgemmParams a; memset(&a, 0, sizeof a);
        a.A = emb; a.B = PP("embed.0.weight"); a.C = e0; a.bias = PP("embed.0.bias"); a.M = B; a.N = E; a.K = ch;
        a.sa_m = ch; a.sa_k = 1; a.sb_k = 1; a.sb_n = ch; a.sc_m = E; a.sc_n = 1; a.alpha = 1.f;
        const dim3 g0((E + 63) / 64, (B + 63) / 64, 1);
        push(fwd_ops, "temb.fc0", 2.0 * B * E * ch, [a, g0](cudaStream_t st) { launch_k(k_sgemm<float, float, float>, g0, 256, 0, st, a); return (int)cudaGetLastError(); });
        SgemmParams b = a; b.A = e0; b.B = PP("embed.2.weight"); b.C = e1; b.bias = PP("embed.2.bias"); b.K = E; b.sa_m = E; b.sb_n = E; b.silu_a = 1; b.ksplit = KS;
        const dim3 g0s((E + 63) / 64, (B + 63) / 64, KS);
        push(fwd_ops, "temb.fc1", 2.0 * B * E * E, [b, g0s](cudaStream_t st) { launch_k(k_sgemm<float, float, float>, g0s, 256, 0, st, b); return (int)cudaGetLastError(); });
        const SgemmParams* tab = at<SgemmParams>(tp_table_off);
        const dim3 g1((maxc + 63) / 64, (B + 63) / 64, nblocks * KS);
        if (tc_temb) {
            // ONE tcgen05 GEMM for all per-block projections: TP[B][tp_ld] = bf16(silu(e1)) x Wcat^T + bias_cat
            const FcEnt* ftab = at<FcEnt>(fc_table_off);
            const dim3 gp(E / 32, maxc / 32, nblocks);
            bf16* WcatT_p = train ? WcatT : nullptr;
            push(pack_ops, "temb.pack_fc", 0, [=](cudaStream_t st) { launch_k(k_pack_fc, gp, dim3(32, 8), 0, st, ftab, Wcat, WcatT_p, bias_cat, E, tp_ld); return (int)cudaGetLastError(); });
            pack_ops.back().wait_pack = 1;
            const long long nE = (long long)B * E;
            push(fwd_ops, "temb.silu_cast", 0, [=](cudaStream_t st) { launch_k(k_cast_bf16, grid_for(nE), 256, 0, st, e1, A_f, nE, 1); return (int)cudaGetLastError(); });
            ddpm_gemm_desc d; memset(&d, 0, sizeof d);
            d.mode = GEMM_KK; d.M = B; d.N = tp_ld; d.W = B; d.H = 1; d.NB = 1;
            d.a_ptr[0] = A_f; d.a_C[0] = E; d.a_ld[0] = E;
            d.nseg = 1; d.seg_map[0] = 0; d.seg_taps[0] = 1; d.seg_kchunks[0] = E / 64; d.seg_cbase[0] = 0;
            d.b_ptr = Wcat; d.b_K = E; d.b_rows = tp_ld; d.b_batch = 1; d.b_ld = E; d.b_bs = 0;
            d.out = TP; d.ldo = tp_ld; d.alpha = 1.f; d.grid_z = 1; d.flags = EPI_OUT_F32; d.bias = bias_cat;
            ++n_tc_gemms;
            if (!dry) {
                GemmLaunch g; const int rc = build_gemm(d, g);
                if (rc) return rc;
                push(fwd_ops, "temb.proj", 0, [g](cudaStream_t st) { return launch_gemm(g, st); });
            } else push(fwd_ops, "temb.proj", 0, [](cudaStream_t) { return 0; });
            fwd_ops.back().wait_pack = 1;
        } else
        push(fwd_ops, "temb.proj", 0, [tab, g1](cudaStream_t st) { launch_k(k_sgemm_table, g1, 256, 0, st, tab, (int)KS); return (int)cudaGetLastError(); });
        fwd_flops += 2.0 * B * E * ch + 2.0 * B * E * E;
        // Sampler steps feed ONE timestep to the whole batch (diffusion.py:166 `t.fill_(ti)`): the embedding MLP and the
        // per-block projections are then computed for a single row and broadcast (ddpm_sampler_step sets uniform_t).
        for (size_t i = temb_first; i < fwd_ops.size(); ++i) fwd_ops[i].tag = OP_TEMB;
        temb_uni_ops.clear();
        push(temb_uni_ops, "temb.sin[1]", 0, [=](cudaStream_t st) { launch_k(k_timestep_embedding, (ch / 2 + 127) / 128, 128, 0, st, self->t_in, emb, 1, ch); return (int)cudaGetLastError(); });
        SgemmParams a1 = a; a1.M = 1; SgemmParams b1 = b; b1.M = 1;
        const dim3 u0((E + 63) / 64, 1, 1), u0s((E + 63) / 64, 1, KS), u1((maxc + 63) / 64, 1, nblocks * KS);
        push(temb_uni_ops, "temb.fc0[1]", 0, [a1, u0](cudaStream_t st) { launch_k(k_sgemm<float, float, float>, u0, 256, 0, st, a1); return (int)cudaGetLastError(); });
        push(temb_uni_ops, "temb.fc1[1]", 0, [b1, u0s](cudaStream_t st) { launch_k(k_sgemm<float, float, float>, u0s, 256, 0, st, b1); return (int)cudaGetLastError(); });
        const SgemmParams* tabu = at<SgemmParams>(tp_uni_table_off);
        push(temb_uni_ops, "temb.proj[1]", 0, [tabu, u1](cudaStream_t st) { launch_k(k_sgemm_table, u1, 256, 0, st, tabu, (int)KS); return (int)cudaGetLastError(); });
        const long long row4 = tp_ld / 4, tot4 = (long long)(Bn - 1) * row4;
        if (Bn > 1 && tp_ld % 4 == 0)
            push(temb_uni_ops, "temb.bcast", 0, [=](cudaStream_t st) { launch_k(k_bcast_rows, (int)((tot4 + 255) / 256), 256, 0, st, reinterpret_cast<float4*>(TP), row4, tot4); return (int)cudaGetLastError(); });
        else if (Bn > 1) temb_uni_ops.clear();     // odd row length: keep the per-row path
    }
    int blk = 0;
    auto tp_entry = [&](const std::string& p, int cout) -> int {
        const int off = blk * maxc; ++blk;
        SgemmParams s; memset(&s, 0, sizeof s);
        s.A = e1; s.B = PP(p + ".fc.weight"); s.C = TP + off; s.bias = PP(p + ".fc.bias"); s.M = B; s.N = cout; s.K = E;
        s.sa_m = E; s.sa_k = 1; s.sb_k = 1; s.sb_n = E; s.sc_m = tp_ld; s.sc_n = 1; s.alpha = 1.f; s.silu_a = 1;
        tp_table_host.push_back(s);
        { SgemmParams u = s; u.M = 1; tp_uni_table_host.push_back(u); }
        { FcEnt f; f.w = PP(p + ".fc.weight"); f.b = PP(p + ".fc.bias"); f.gw = train ? GP(p + ".fc.weight") : nullptr; f.cout = cout; f.off = off; fc_table_host.push_back(f); }
        fwd_flops += 2.0 * B * cout * E;
        if (train) {
            // dW_fc[o][e] = sum_b silu(e1[b][e]) * dTP[b][off+o]   (computed as C'[e][o], stored transposed)
            SgemmParams w; memset(&w, 0, sizeof w);
            w.A = e1; w.B = dTP + off; w.C = GP(p + ".fc.weight"); w.M = E; w.N = cout; w.K = B;
            w.sa_m = 1; w.sa_k = E; w.sb_k = tp_ld; w.sb_n = 1; w.sc_m = 1; w.sc_n = E; w.alpha = 1.f; w.silu_a = 1;
            tpw_table_host.push_back(w);
            // d_st[b][e] += sum_o dTP[b][off+o] * W_fc[o][e]
            SgemmParams d; memset(&d, 0, sizeof d);
            d.A = dTP + off; d.B = PP(p + ".fc.weight"); d.C = d_st; d.M = B; d.N = E; d.K = cout;
            d.sa_m = tp_ld; d.sa_k = 1; d.sb_k = E; d.sb_n = 1; d.sc_m = E; d.sc_n = 1; d.alpha = 1.f; d.accumulate = 2;
            tpd_table_host.push_back(d);
            bwd_flops += 4.0 * B * cout * E;
        }
        return off;
    };
    if (train) {
        // adjoint of the embedding MLP; registered first so it runs after every block has deposited its dTP slice
        tape_push([=]() {
            const SgemmParams* tw = at<SgemmParams>(tpw_table_off); const SgemmParams* td = at<SgemmParams>(tpd_table_off);
            const dim3 gw((maxc + 63) / 64, (E + 63) / 64, nblocks), gd((E + 63) / 64, (B + 63) / 64, nblocks);
            if (tc_temb) {
                // dTP -> bf16 once; dW_cat [tp_ld][E] = dTP^T x silu(e1) (MN-major GEMM) scattered to the 22 fc.weight grads;
                // d_st [B][E] = dTP x Wcat (K-major GEMM over K = tp_ld, split-K atomics into the zeroed d_st)
                bf16* dTPb = at<bf16>(alloc((size_t)B * tp_ld * 2));
                float* Sw = at<float>(alloc((size_t)tp_ld * E * 4));
                const long long nT = (long long)B * tp_ld;
                const FcEnt* ftab = at<FcEnt>(fc_table_off);
                push(bwd_ops, "temb.dtp_cast", 0, [=](cudaStream_t st) { launch_k(k_cast_bf16, grid_for(nT), 256, 0, st, dTP, dTPb, nT, 0); return (int)cudaGetLastError(); });
                ddpm_gemm_desc w; memset(&w, 0, sizeof w);
                w.mode = GEMM_MNMN; w.M = tp_ld; w.N = E; w.W = B; w.H = 1; w.NB = 1;
                w.a_ptr[0] = dTPb; w.a_C[0] = tp_ld; w.a_ld[0] = tp_ld;
                w.b_ptr = A_f; w.b_K = E; w.b_ld = E;
                w.taps = 1; w.kblocks = B / 64; w.splits = 1; w.grid_z = 1;
                w.flags = EPI_OUT_F32; w.alpha = 1.f; w.out = Sw; w.ldo = E;
                ddpm_gemm_desc d; memset(&d, 0, sizeof d);
                d.mode = GEMM_KK; d.M = B; d.N = E; d.W = B; d.H = 1; d.NB = 1;
                d.a_ptr[0] = dTPb; d.a_C[0] = tp_ld; d.a_ld[0] = tp_ld;
                d.nseg = 1; d.seg_map[0] = 0; d.seg_taps[0] = 1; d.seg_kchunks[0] = tp_ld / 64; d.seg_cbase[0] = 0;
                d.b_ptr = WcatT; d.b_K = tp_ld; d.b_rows = E; d.b_batch = 1; d.b_ld = tp_ld; d.b_bs = 0;
                const int n_t = (E + 255) / 256; int ks = 148 / n_t; if (ks > tp_ld / 64 / 4) ks = tp_ld / 64 / 4; if (ks > 32) ks = 32; if (ks < 1) ks = 1;
                d.kk_splits = ks; d.grid_z = ks; d.out = d_st; d.ldo = E; d.alpha = 1.f; d.flags = EPI_OUT_F32 | EPI_ATOMIC;
                n_tc_gemms += 2;
                const dim3 gsc((unsigned)(((long long)maxc * E / 4 + 255) / 256), nblocks);
                if (!dry) {
                    GemmLaunch gwl, gdl; int rc = build_gemm(w, gwl); if (!rc) rc = build_gemm(d, gdl);
                    if (rc) { plan_error = rc; return; }
                    push(bwd_ops, "temb.proj.bwd", 0, [=](cudaStream_t st) {
                        int r = launch_gemm(gwl, st); if (r) return r;
                        launch_k(k_scatter_fc_grad, gsc, 256, 0, st, ftab, reinterpret_cast<const float4*>(Sw), E);
                        r = launch_gemm(gdl, st); if (r) return r;
                        return (int)cudaGetLastError(); }, 3);
                } else push(bwd_ops, "temb.proj.bwd", 0, [](cudaStream_t) { return 0; }, 3);
            } else
            push(bwd_ops, "temb.proj.bwd", 0, [=](cudaStream_t st) { launch_k(k_sgemm_table, gw, 256, 0, st, tw, 1); launch_k(k_sgemm_table, gd, 256, 0, st, td, 1); return (int)cudaGetLastError(); }, 2);
            float* d_e1 = at<float>(alloc((size_t)B * E * 4)); float* d_s0 = at<float>(zero_bwd((size_t)B * E * 4)); float* d_e0 = at<float>(alloc((size_t)B * E * 4));
            const long long nE = (long long)B * E; const int Bn = B;
            float* gw2 = GP("embed.2.weight"); float* gb2 = GP("embed.2.bias"); float* gw0 = GP("embed.0.weight"); float* gb0 = GP("embed.0.bias");
            const float* w2 = PP("embed.2.weight");
            push(bwd_ops, "temb.mlp.bwd", 0, [=](cudaStream_t st) {
                launch_k(k_silu_bwd_f32, grid_for(nE), 256, 0, st, e1, d_st, d_e1, nE);
                SgemmParams a; memset(&a, 0, sizeof a);           // dW2[n][k] = sum_b silu(e0[b][k]) d_e1[b][n]
                a.A = e0; a.B = d_e1; a.C = gw2; a.M = E; a.N = E; a.K = Bn; a.sa_m = 1; a.sa_k = E; a.sb_k = E; a.sb_n = 1; a.sc_m = 1; a.sc_n = E; a.alpha = 1.f; a.silu_a = 1;
                launch_k(k_sgemm<float, float, float>, dim3((E + 63) / 64, (E + 63) / 64, 1), 256, 0, st, a);
                launch_k(k_colsum_f32, (E + 127) / 128, 128, 0, st, d_e1, gb2, Bn, E, E);
                SgemmParams b; memset(&b, 0, sizeof b);           // d_s0[b][k] = sum_n d_e1[b][n] W2[n][k]
                b.A = d_e1; b.B = w2; b.C = d_s0; b.M = Bn; b.N = E; b.K = E; b.sa_m = E; b.sa_k = 1; b.sb_k = E; b.sb_n = 1; b.sc_m = E; b.sc_n = 1; b.alpha = 1.f; b.ksplit = 4;
                launch_k(k_sgemm<float, float, float>, dim3((E + 63) / 64, (Bn + 63) / 64, 4), 256, 0, st, b);
                launch_k(k_silu_bwd_f32, grid_for(nE), 256, 0, st, e0, d_s0, d_e0, nE);
                SgemmParams c; memset(&c, 0, sizeof c);           // dW0[n][k] = sum_b emb[b][k] d_e0[b][n]
                c.A = emb; c.B = d_e0; c.C = gw0; c.M = ch; c.N = E; c.K = Bn; c.sa_m = 1; c.sa_k = ch; c.sb_k = E; c.sb_n = 1; c.sc_m = 1; c.sc_n = ch; c.alpha = 1.f;
                launch_k(k_sgemm<float, float, float>, dim3((E + 63) / 64, (ch + 63) / 64, 1), 256, 0, st, c);
                launch_k(k_colsum_f32, (E + 127) / 128, 128, 0, st, d_e0, gb0, Bn, E, E);
                return (int)cudaGetLastError(); }, 7);
        });
    }

    // ---- in_conv (unet.py:127,210): NCHW fp32 -> NHWC bf16
    cur_tag = "d0";
    T4 h0 = newT(B, H, W, ch);
    {
        const float* wi = PP("in_conv.weight"); const float* bi = PP("in_conv.bias"); bf16* o = bp(h0);
        const size_t shm = (size_t)(ch * Cin * 9 + ch) * 4; const int n = grid_for((long long)B * H * W / 2, 128);
        const int Bn = B, Hn = H, Wn = W;
        // h0 feeds the first norm1 and (as the last skip) the final up block's norm1: its statistics come out of this kernel
        double* qs0 = nullptr;
        if (ch % 32 == 0 && (H * W) % 32 == 0 && !getenv("DDPM_NO_GN_EPI")) { h0.qs = (long long)zero_fwd((size_t)B * (ch / 4) * 2 * 8); qs0 = at<double>((size_t)h0.qs); }
        // tensor-core route: X = im2col(x) [P][KP] bf16 (9*Cin patch columns, zero padded to whole K slabs: KP = 64 up to 7
        // channels, 128 / 192 for 8..16) and a 1x1 "conv" over it; the training backward reuses X for the weight gradient.
        // (CUDA-core k_in_conv otherwise, up to 4 channels.)
        static const bool no_tc_inconv = getenv("DDPM_NO_TC_INCONV") != nullptr;
        const bool tc_in = wide_in || (!no_tc_inconv && ch % 64 == 0 && tc_ok_geom(H, W) && Cin <= 4);
        const int KP = im2col_width(Cin);
        T4 Xcol;
        if (tc_in) {
            Xcol = newT(B, H, W, KP);
            bf16* Xp = bp(Xcol);
            bf16* wpk = at<bf16>(alloc((size_t)ch * KP * 2));
            const int npk = (ch * KP + 255) / 256; const int chn = ch, cin = Cin;
            push(pack_ops, "in_conv.pack", 0, [=](cudaStream_t st) { launch_k(k_pack_in, npk, 256, 0, st, wi, wpk, chn, cin, KP); return (int)cudaGetLastError(); });
            pack_ops.back().wait_pack = 1;             // "early" pack: in_conv is the first consumer of the forward pass
            const int nim = grid_for((long long)B * H * W);
            push(fwd_ops, "in_conv.im2col", 0, [=](cudaStream_t st) {
                // training: x_t = q_sample(x0, t, noise) is formed while the patches are gathered
                launch_im2col3(cin, nim, st, self->x_in, Xp, Bn, Hn, Wn, 1, self->qs_pro);
                return (int)cudaGetLastError(); });
            ConvSpec c; c.name = "in_conv"; c.in = one(Xcol); c.ksize = 1; c.wp = wpk; c.ldw = KP; c.bias = bi; c.out = h0; c.Co = ch; c.Ho = H; c.Wo = W;
            c.want_qstats = true;
            const size_t first_conv = fwd_ops.size();
            h0.qs = conv_op(fwd_ops, c, nullptr);
            if (first_conv < fwd_ops.size()) fwd_ops[first_conv].wait_pack = 1;
        } else
        push(fwd_ops, "in_conv", 2.0 * B * H * W * ch * Cin * 9, [=](cudaStream_t st) {
            const QsamplePro qp = self->qs_pro;       // training: x_t = q_sample(x0, t, noise) is formed while the taps are loaded
            switch (Cin) {
                case 1: launch_k(k_in_conv<1>, n, 128, shm, st, self->x_in, wi, bi, o, Bn, Hn, Wn, ch, qs0, qp); break;
                case 2: launch_k(k_in_conv<2>, n, 128, shm, st, self->x_in, wi, bi, o, Bn, Hn, Wn, ch, qs0, qp); break;
                case 3: launch_k(k_in_conv<3>, n, 128, shm, st, self->x_in, wi, bi, o, Bn, Hn, Wn, ch, qs0, qp); break;
                default: launch_k(k_in_conv<4>, n, 128, shm, st, self->x_in, wi, bi, o, Bn, Hn, Wn, ch, qs0, qp); break;
            }
            return (int)cudaGetLastError(); });
        fwd_flops += 2.0 * B * H * W * ch * Cin * 9;
        first_packed_op = fwd_ops.size();          // in_conv reads the fp32 master weights; everything after it reads packed ones
        if (train) tape_push([=]() {
            const T4 dY = grad_of(h0, nullptr);
            float* gw = GP("in_conv.weight"); float* gb = GP("in_conv.bias"); const bf16* d = bp(dY);
            const long long P = (long long)Bn * Hn * Wn; const int ppb = 256; const int nb = (int)((P + ppb - 1) / ppb);
            bwd_flops += 2.0 * P * ch * Cin * 9;
            const long long s_c = (long long)Cin * 9;
            static const bool no_tc_in = getenv("DDPM_NO_TC_OUTCONV") != nullptr;
            if (wide_in || (!no_tc_in && ch % 64 == 0 && tc_ok_geom(H, W) && 9 * Cin <= 64)) {
                // weight gradient on the tensor cores: X = im2col(x) [P][KP] bf16, S[ch][KP] = dY^T x X (MN-major GEMM, side stream)
                T4 X = tc_in ? Xcol : newT(B, H, W, KP);
                bf16* Xp = bp(X);
                const int nim = grid_for(P);
                if (!tc_in) push(bwd_ops, "in_conv.im2col", 0, [=](cudaStream_t st) {
                    launch_im2col3(Cin, nim, st, self->x_in, Xp, Bn, Hn, Wn, 1, QsamplePro{nullptr, nullptr, nullptr, nullptr, nullptr});
                    return (int)cudaGetLastError(); }, 1, true);
                float* S2 = at<float>(zero_bwd((size_t)ch * KP * 4));
                wgrad_op("in_conv.wgrad", dY, one(X), 1, 1, MAP_NORMAL, S2, ch);
                const int nun = (ch * Cin * 9 + 255) / 256;
                push(bwd_ops, "in_conv.wunpack", 0, [=](cudaStream_t st) { launch_k(k_unpack_tap, nun, 256, 0, st, S2, gw, ch, Cin, 1, KP); return (int)cudaGetLastError(); }, 1, true);
                colsum_op("in_conv.bias", dY, nullptr, 0, gb, nullptr, ch);
                return;
            }
            push(bwd_ops, "in_conv.wgrad", 2.0 * P * ch * Cin * 9, [=](cudaStream_t st) {
                switch (Cin) {
                    case 1: launch_k(k_corr3x3<1>, nb, ch, 0, st, d, self->x_in, gw, s_c, 9, 1, 0, gb, Bn, Hn, Wn, ch, ppb); break;
                    case 2: launch_k(k_corr3x3<2>, nb, ch, 0, st, d, self->x_in, gw, s_c, 9, 1, 0, gb, Bn, Hn, Wn, ch, ppb); break;
                    case 3: launch_k(k_corr3x3<3>, nb, ch, 0, st, d, self->x_in, gw, s_c, 9, 1, 0, gb, Bn, Hn, Wn, ch, ppb); break;
                    default: launch_k(k_corr3x3<4>, nb, ch, 0, st, d, self->x_in, gw, s_c, 9, 1, 0, gb, Bn, Hn, Wn, ch, ppb); break;
                }
                return (int)cudaGetLastError(); });
        });
    }

    // ---- down path (unet.py:210-218)
    std::vector<T4> hs; hs.push_back(h0);
    auto block = [&](const std::string& p, const Src& x, int cout, bool at_) -> T4 {
        if (at_) { const int off = tp_entry(p + ".0", cout); T4 r = res_block(p + ".0", x, cout, off, tp_ld, TP, dTP); return attn_block(p + ".1", r); }
        const int off = tp_entry(p, cout); return res_block(p, x, cout, off, tp_ld, TP, dTP);
    };
    for (int i = 0; i < L; ++i) {
        const std::string p = "downsamples.level_" + std::to_string(i);
        cur_tag = "d" + std::to_string(i);
        for (int j = 0; j < nrb; ++j) hs.push_back(block(p + "." + std::to_string(j), one(hs.back()), chs(i), cfg.attn[i] != 0));
        if (i != L - 1) hs.push_back(down_conv(p + "." + std::to_string(nrb) + ".1", hs.back()));
    }
    // ---- middle (unet.py:132-136,221)
    T4 h = hs.back();
    cur_tag = "mid";
    { const int off = tp_entry("middle.0", chs(L - 1)); h = res_block("middle.0", one(h), chs(L - 1), off, tp_ld, TP, dTP); }
    h = attn_block("middle.1", h);
    { const int off = tp_entry("middle.2", chs(L - 1)); h = res_block("middle.2", one(h), chs(L - 1), off, tp_ld, TP, dTP); }
    // ---- up path (unet.py:224-230): cat([h, hs.pop()]) is never materialised
    for (int i = L - 1; i >= 0; --i) {
        const std::string p = "upsamples.level_" + std::to_string(i);
        cur_tag = "u" + std::to_string(i);
        for (int j = 0; j <= nrb; ++j) {
            Src s; s.t0 = h; s.t1 = hs.back(); s.two = true; hs.pop_back();
            h = block(p + "." + std::to_string(j), s, chs(i), cfg.attn[i] != 0);
        }
        if (i != 0) h = up_conv(p + "." + std::to_string(nrb + 1) + ".1", h);
    }
    if (blk != nblocks) return fail(-31, "internal: block count mismatch %d vs %d", blk, nblocks);
    // ---- out_conv (unet.py:138-142,232): GN -> SiLU -> conv3x3 (C -> Cout<=16) -> NCHW fp32
    cur_tag = "u" + std::to_string(L - 1);           // its parameters sit right behind upsamples.level_{L-1} in the flat buffer
    {
        if (ch > 256) return fail(-30, "hid_channels > 256 unsupported by the narrow out_conv kernels");
        T4 a_out = newT(B, H, W, ch);
        const GnSaved g = gn_fwd(fwd_ops, "out_conv.0", one(h), "out_conv.0", a_out, 1, 0.f);
        const float* wo = PP("out_conv.2.weight"); const float* bo = PP("out_conv.2.bias"); const bf16* ap = bp(a_out);
        const int Bn = B, Hn = H, Wn = W;
        const size_t shm = (size_t)9 * Cout * ch * 4;
        if (W % 4) return fail(-30, "image width must be a multiple of 4");
        const int nblk = grid_for((long long)B * H * W);
        const double fl = 2.0 * B * H * W * ch * Cout * 9;
        fwd_flops += fl;
        static const bool no_tc_out = getenv("DDPM_NO_TC_OUTCONV") != nullptr;
        bool tc_out = wide_out || (!no_tc_out && ch % 64 == 0 && tc_ok_geom(H, W) && 9 * Cout <= 32);
        // tap-output width of the forward GEMM (32 up to 3 channels, 64 / 128 / 192 for 5..16) and patch width of the backward's im2col
        const int TW = tap_width(Cout), KPo = im2col_width(Cout);
        bf16* w27t = nullptr;
        if (tc_out) {
            // tensor-core path: 1x1 GEMM a[P][ch] x W27[TW][ch]^T -> fp32 tap outputs T[P][TW], then a 9-point gather
            bf16* w27 = at<bf16>(alloc_once_zero((size_t)TW * ch * 2));
            float* T = at<float>(alloc((size_t)B * H * W * TW * 4));
            const int npk = (Cout * ch * 9 + 255) / 256;
            push(pack_ops, "out_conv.pack27", 0, [=](cudaStream_t st) { launch_k(k_pack_tapco, npk, 256, 0, st, wo, w27, Cout, ch); return (int)cudaGetLastError(); });
            if (train) {
                w27t = at<bf16>(alloc_once_zero((size_t)ch * KPo * 2));
                bf16* w27tp = w27t;
                push(pack_ops, "out_conv.pack27t", 0, [=](cudaStream_t st) { launch_k(k_pack_tapco_t, npk, 256, 0, st, wo, w27tp, Cout, ch, KPo); return (int)cudaGetLastError(); });
            }
            ddpm_gemm_desc d; memset(&d, 0, sizeof d);
            d.mode = GEMM_KK; d.M = B * H * W; d.N = TW; d.block_n = 64; d.W = W; d.H = H; d.NB = B;
            d.a_ptr[0] = ap; d.a_C[0] = ch; d.a_ld[0] = ch;
            d.nseg = 1; d.seg_map[0] = 0; d.seg_taps[0] = 1; d.seg_kchunks[0] = ch / 64; d.seg_cbase[0] = 0;
            d.b_ptr = w27; d.b_K = ch; d.b_rows = TW; d.b_batch = 1; d.b_ld = ch; d.b_bs = 0;
            d.out = T; d.ldo = TW; d.alpha = 1.f; d.grid_z = 1; d.flags = EPI_OUT_F32;
            ++n_tc_gemms;
            if (!dry) {
                GemmLaunch g; const int rc = build_gemm(d, g);
                if (rc) return rc;
                push(fwd_ops, "out_conv.2", fl, [g](cudaStream_t st) { return launch_gemm(g, st); });
            } else push(fwd_ops, "out_conv.2", fl, [](cudaStream_t) { return 0; });
            gather_fused_tail = true;             // the sampler's alpha/beta update rides in this kernel (ddpm_sampler_step)
            push(fwd_ops, "out_conv.2.gather", 0, [=](cudaStream_t st) {
                launch_out_gather(Cout, nblk, st, T, bo, self->eps_dst, Bn, Hn, Wn, self->ps_epi);
                return (int)cudaGetLastError(); });
        } else
        push(fwd_ops, "out_conv.2", fl, [=](cudaStream_t st) {
            switch (Cout) {
                case 1: launch_k(k_out_conv<1>, nblk, 256, shm, st, ap, wo, bo, self->eps_dst, Bn, Hn, Wn, ch); break;
                case 2: launch_k(k_out_conv<2>, nblk, 256, shm, st, ap, wo, bo, self->eps_dst, Bn, Hn, Wn, ch); break;
                case 3: launch_k(k_out_conv<3>, nblk, 256, shm, st, ap, wo, bo, self->eps_dst, Bn, Hn, Wn, ch); break;
                default: launch_k(k_out_conv<4>, nblk, 256, shm, st, ap, wo, bo, self->eps_dst, Bn, Hn, Wn, ch); break;
            }
            return (int)cudaGetLastError(); });
        if (train) {
            // data gradient = a 3x3 "in_conv" Cout -> ch over d_eps with flipped / transposed fp32 weights
            float* wt = at<float>(alloc((size_t)ch * Cout * 9 * 4));
            { PackEntry e; memset(&e, 0, sizeof e); e.kind = PK_FLIP_T; e.Co = Cout; e.Ci = ch; e.taps = 9; e.w = wo; e.fout = wt; pack_table_host.push_back(e); }
            tape_push([=]() {
                float* gw = GP("out_conv.2.weight"); float* gb = GP("out_conv.2.bias");
                T4 d_a = newT(B, H, W, ch);
                bf16* dap = bp(d_a);
                const size_t shm2 = (size_t)(ch * Cout * 9 + ch) * 4; const int n2 = grid_for((long long)Bn * Hn * Wn / 2, 128);
                const long long P = (long long)Bn * Hn * Wn; const int ppb = 256; const int nb = (int)((P + ppb - 1) / ppb);
                bwd_flops += 2.0 * fl;
                if (tc_out) {
                    // tensor-core backward: E = im2col(d_eps) [P][KPo] bf16 (shared by both gradients);
                    // d_a = E x W27^T (1x1 conv KPo -> ch), dW = E^T x a (MN-major GEMM on the side stream) -> OIHW
                    T4 E = newT(B, H, W, KPo);
                    bf16* Ep = bp(E);
                    const int nim = grid_for((long long)Bn * Hn * Wn);
                    push(bwd_ops, "out_conv.2.im2col", 0, [=](cudaStream_t st) {
                        const float* de = self->deps_src;
                        launch_k(k_chansum_nchw, dim3(64, Cout), 256, 0, st, de, gb, Bn, Cout, Hn * Wn);
                        launch_im2col3(Cout, nim, st, de, Ep, Bn, Hn, Wn, -1, QsamplePro{nullptr, nullptr, nullptr, nullptr, nullptr});
                        return (int)cudaGetLastError(); }, 2);
                    ConvSpec cs; cs.name = "out_conv.2.dgrad"; cs.in = one(E); cs.ksize = 1; cs.wp = w27t; cs.ldw = KPo;
                    cs.out = d_a; cs.Co = ch; cs.Ho = H; cs.Wo = W;
                    conv_op(bwd_ops, cs, nullptr);
                    float* S = at<float>(zero_bwd((size_t)KPo * ch * 4));
                    wgrad_op("out_conv.2.wgrad", E, one(a_out), 1, 1, MAP_NORMAL, S, KPo);
                    const int nun = (Cout * ch * 9 + 255) / 256;
                    push(bwd_ops, "out_conv.2.wunpack", 0, [=](cudaStream_t st) { launch_k(k_unpack_tap, nun, 256, 0, st, S, gw, Cout, ch, 0, KPo); return (int)cudaGetLastError(); }, 1, true);
                } else
                push(bwd_ops, "out_conv.2.bwd", 2.0 * fl, [=](cudaStream_t st) {
                    const float* de = self->deps_src;
                    launch_k(k_chansum_nchw, dim3(64, Cout), 256, 0, st, de, gb, Bn, Cout, Hn * Wn);
                    switch (Cout) {
                        case 1: launch_k(k_in_conv<1>, n2, 128, shm2, st, de, wt, nullptr, dap, Bn, Hn, Wn, ch, (double*)nullptr, QsamplePro{});
                                launch_k(k_corr3x3<1>, nb, ch, 0, st, ap, de, gw, 9, (long long)ch * 9, 1, 1, nullptr, Bn, Hn, Wn, ch, ppb); break;
                        case 2: launch_k(k_in_conv<2>, n2, 128, shm2, st, de, wt, nullptr, dap, Bn, Hn, Wn, ch, (double*)nullptr, QsamplePro{});
                                launch_k(k_corr3x3<2>, nb, ch, 0, st, ap, de, gw, 9, (long long)ch * 9, 1, 1, nullptr, Bn, Hn, Wn, ch, ppb); break;
                        case 3: launch_k(k_in_conv<3>, n2, 128, shm2, st, de, wt, nullptr, dap, Bn, Hn, Wn, ch, (double*)nullptr, QsamplePro{});
                                launch_k(k_corr3x3<3>, nb, ch, 0, st, ap, de, gw, 9, (long long)ch * 9, 1, 1, nullptr, Bn, Hn, Wn, ch, ppb); break;
                        default: launch_k(k_in_conv<4>, n2, 128, shm2, st, de, wt, nullptr, dap, Bn, Hn, Wn, ch, (double*)nullptr, QsamplePro{});
                                launch_k(k_corr3x3<4>, nb, ch, 0, st, ap, de, gw, 9, (long long)ch * 9, 1, 1, nullptr, Bn, Hn, Wn, ch, ppb); break;
                    }
                    return (int)cudaGetLastError(); }, 3);
                gn_bwd("out_conv.0", g, d_a, nullptr);
            });
        }
    }
    // ---- backward list: zero accumulators + flat grads, then the tape in reverse
    if (train) {
        uint8_t* z = ws + zero_bwd_off; const size_t n = zero_bwd_bytes; float* Gp = G; const size_t gbytes = (size_t)flat_elems * 4;
        push(bwd_ops, "zero.bwd", 0, [=](cudaStream_t st) {
            if (n) { const cudaError_t e = cudaMemsetAsync(z, 0, n, st); if (e) return (int)e; }
            return (int)cudaMemsetAsync(Gp, 0, gbytes, st); }, 0);
        // the tape in reverse; whenever every entry of a level group has run, its slice of the flat gradient buffer is final:
        // groups are merged into chunks of >= 4 M gradients (16 MB) as long as they stay contiguous, and every chunk boundary
        // becomes an op that unpacks the chunk's weight gradients on the side stream and records the chunk's event
        std::map<std::string, std::pair<long long, long long>> range;
        for (auto& pr : params) {
            const std::string g = group_of(pr.name);
            const long long lo = pr.off, hi = pr.off + (pr.numel + 63) / 64 * 64;
            auto it = range.find(g);
            if (it == range.end()) range[g] = {lo, hi}; else { if (lo < it->second.first) it->second.first = lo; if (hi > it->second.second) it->second.second = hi; }
        }
        std::map<std::string, int> remaining;
        for (auto& tg : tape_tag) ++remaining[tg];
        // the table must exist before the ops are built: its size is only known after the tape ran, so reserve the worst case
        const size_t max_unpack = 2 * params.size() + 8;
        unpack_table_off = alloc(sizeof(PackEntry) * max_unpack);
        const PackEntry* tab = at<PackEntry>(unpack_table_off);
        long long pend_lo = -1, pend_hi = -1; int unpack_done = 0;
        auto emit = [&]() {
            if (pend_lo < 0) return;
            GradChunk c; c.lo = pend_lo; c.hi = pend_hi; c.unpack_lo = unpack_done; c.unpack_hi = (int)unpack_table_host.size();
            unpack_done = c.unpack_hi;
            const int idx = (int)chunks.size();
            chunks.push_back(c);
            const int n = c.unpack_hi - c.unpack_lo; const PackEntry* t0 = tab + c.unpack_lo;
            Op o; o.name = "grad.chunk" + std::to_string(idx); o.flops = 0; o.launches = n > 0 ? 1 : 0; o.chunk = idx;
            o.run = [=](cudaStream_t st) { if (n > 0) { launch_k(k_pack_table, dim3(128, n), 256, 0, st, t0); return (int)cudaGetLastError(); } return 0; };
            bwd_ops.push_back(std::move(o));
            pend_lo = pend_hi = -1;
        };
        for (int i = (int)tape.size() - 1; i >= 0; --i) {
            tape[i]();
            const std::string& tg = tape_tag[i];
            if (--remaining[tg] > 0) continue;
            auto it = range.find(tg);
            if (it == range.end()) continue;
            const long long lo = it->second.first, hi = it->second.second;
            if (pend_lo >= 0 && !(lo == pend_hi || hi == pend_lo)) emit();          // not adjacent: close the pending chunk first
            if (pend_lo < 0) { pend_lo = lo; pend_hi = hi; } else { if (lo < pend_lo) pend_lo = lo; if (hi > pend_hi) pend_hi = hi; }
            if (pend_hi - pend_lo >= (4 << 20) || tg == "late") emit();
        }
        emit();
        if (unpack_table_host.size() > max_unpack) return fail(-31, "internal: gradient unpack table overflow");
        tape.clear();
    }
    pack_table_off = alloc(sizeof(PackEntry) * (pack_table_host.size() + 1));
    if (!pack_table_host.empty()) {
        const PackEntry* tab = at<PackEntry>(pack_table_off); const int n = (int)pack_table_host.size();
        push(pack_ops, "pack_all", 0, [=](cudaStream_t st) { launch_k(k_pack_table, dim3(128, n), 256, 0, st, tab); return (int)cudaGetLastError(); });
    }
    if (plan_error) return plan_error;
    return 0;
}

inline int UnetEngine::build() {
    // a re-plan moves the workspace offsets: a weight re-pack of the PREVIOUS plan that is still queued on the (non-blocking) side
    // stream must have drained before the tables are rewritten and before the new plan's first ops touch the workspace
    if (side_stream) cudaStreamSynchronize(side_stream);
    pack_pending = false;
    // tables -> device ; plan-time zeroed arenas
    auto up = [&](size_t off, const std::vector<SgemmParams>& v) -> int {
        if (v.empty()) return 0;
        return (int)cudaMemcpy(ws + off, v.data(), v.size() * sizeof(SgemmParams), cudaMemcpyHostToDevice);
    };
    int rc;
    if ((rc = up(tp_uni_table_off, tp_uni_table_host))) return rc;
    if (!fc_table_host.empty() && cudaMemcpy(ws + fc_table_off, fc_table_host.data(), fc_table_host.size() * sizeof(FcEnt), cudaMemcpyHostToDevice))
        return fail(-2, "fc table upload failed");
    if ((rc = up(tp_table_off, tp_table_host)) || (rc = up(tpw_table_off, tpw_table_host)) || (rc = up(tpd_table_off, tpd_table_host)))
        return fail(-2, "table upload failed: %s", cudaGetErrorString((cudaError_t)rc));
    if (!pack_table_host.empty() && cudaMemcpy(ws + pack_table_off, pack_table_host.data(), pack_table_host.size() * sizeof(PackEntry), cudaMemcpyHostToDevice))
        return fail(-2, "pack table upload failed");
    if (!unpack_table_host.empty() && cudaMemcpy(ws + unpack_table_off, unpack_table_host.data(), unpack_table_host.size() * sizeof(PackEntry), cudaMemcpyHostToDevice))
        return fail(-2, "unpack table upload failed");
    for (auto& r : once_list) { const cudaError_t e = cudaMemset(ws + r.first, 0, r.second); if (e) return fail(-2, "memset failed: %s", cudaGetErrorString(e)); }
    if (!side_stream) {
        if (cudaStreamCreateWithFlags(&side_stream, cudaStreamNonBlocking) || cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming) ||
            cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming)) return fail(-2, "side stream creation failed");
        if (cudaEventCreateWithFlags(&ev_pack_fork, cudaEventDisableTiming) || cudaEventCreateWithFlags(&ev_pack_fc, cudaEventDisableTiming) ||
            cudaEventCreateWithFlags(&ev_pack_all, cudaEventDisableTiming)) return fail(-2, "repack event creation failed");
    }
    if (first_packed_op < fwd_ops.size()) fwd_ops[first_packed_op].wait_pack = 2;
    for (auto& c : chunks)
        if (!c.ev && cudaEventCreateWithFlags(&c.ev, cudaEventDisableTiming)) return fail(-2, "gradient-chunk event creation failed");
    planned = true;
    return 0;
}

}  // namespace ddpm
