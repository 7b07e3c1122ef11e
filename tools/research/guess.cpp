// guess.cpp — multiple shooting from an INFORMED guess: entry heads of every segment from an occupancy scan (what is conserved:
// quads taken, slices filled) + a time-balanced split inside a trading group, then absolute chaining (entry(s+1) = end(s)).
//   ./guess <c3|c4> <segment GPUs> [warm-up GPUs]
#include "shoot_common.cpp"
#include <cmath>
static int psize(int p) { return profs[p].masks.empty() ? 0 : __builtin_popcount(profs[p].masks[0]); }
// number of requests of profile p with time < tau
static uint32_t cnt_before(int p, uint32_t tau) { return std::lower_bound(q[p].begin(), q[p].end(), tau) - q[p].begin(); }

int main(int argc, char** argv) {
    const std::string cfg = argc > 1 ? argv[1] : "c4";
    const uint32_t seg = argc > 2 ? atoi(argv[2]) : 512;
    const bool newton = argc > 3 ? atoi(argv[3]) : 0;
    Loaded L = load_config(cfg);
    const uint32_t G = L.occ.size(), S = (G + seg - 1) / seg;
    size_t off = 0;
    for (size_t b = 0; b < L.sizes.size() && b < 16; ++b) {
        const uint32_t n = L.sizes[b];
        open_batch(L, off, n);
        const int np = (int)profs.size();
        std::vector<Heads> truth(S + 1); Heads h0{}; truth[0] = h0;
        std::vector<uint8_t> occ_new = L.occ; uint64_t dec = 0;
        for (uint32_t s = 0; s < S; ++s) truth[s + 1] = simulate(L.occ, s * seg, std::min(G, (s + 1) * seg), truth[s], &dec, &occ_new);
        // ---- the guess
        std::vector<int> big, small;          // size >= 4 group / size 1,2 group
        for (int p = 0; p < np; ++p) { int sz = psize(p); if (!sz || q[p].empty()) continue; if (sz >= 4) big.push_back(p); else small.push_back(p); }
        uint64_t totbig = 0; for (int p : big) totbig += q[p].size();
        uint64_t totsmall_mass = 0; for (int p : small) totsmall_mass += (uint64_t)q[p].size() * psize(p);
        uint32_t usable1 = 0; for (int p : small) for (uint32_t m : profs[p].masks) usable1 |= m;
        std::vector<Heads> H(S + 1, h0);
        uint64_t Q = 0, R = 0;
        for (uint32_t g = 0; g <= G; ++g) {
            if (g % seg == 0 || g == G) {
                const uint32_t s = g == G ? S : g / seg;
                Heads h{};
                // big group: first Q of the merged queue
                { uint32_t lo = 0, hi = n; while (lo < hi) { uint32_t mid = (lo + hi) / 2; uint64_t c = 0; for (int p : big) c += cnt_before(p, mid); if (c >= Q) hi = mid; else lo = mid + 1; }
                  for (int p : big) h[p] = cnt_before(p, lo); }
                // small group: balanced time
                { uint32_t lo = 0, hi = n; while (lo < hi) { uint32_t mid = (lo + hi) / 2; uint64_t c = 0; for (int p : small) c += (uint64_t)cnt_before(p, mid) * psize(p); if (c >= R) hi = mid; else lo = mid + 1; }
                  for (int p : small) h[p] = cnt_before(p, lo); }
                if (getenv("PROPG")) {
                    uint64_t nb = 0, ns = 0; for (int p : big) nb += q[p].size(); for (int p : small) ns += (uint64_t)q[p].size() * psize(p);
                    for (int p : big) h[p] = std::min<uint64_t>(q[p].size(), nb ? (Q * q[p].size() + nb / 2) / nb : 0);
                    for (int p : small) h[p] = std::min<uint64_t>(q[p].size(), ns ? (R * q[p].size() + ns / 2) / ns : 0);
                }
                if (s <= S) H[s] = h;
                if (g == G) break;
            }
            uint32_t o = L.occ[g];
            if (Q < totbig) { for (int p : big) { bool took = false; for (uint32_t m : profs[p].masks) if (!(o & m)) { o |= m; ++Q; took = true; break; } if (took) break; } }
            if (R < totsmall_mass) R += __builtin_popcount(~o & usable1);
        }
        H[0] = h0;
        // ---- error of the guess
        { double e1 = 0, e2 = 0; int busy = 0; long maxabs = 0;
          for (uint32_t s = 1; s < S; ++s) { if (truth[s] == truth[s + 1] && s > 1) continue; ++busy;
              long dq = 0, dr = 0; for (int p : big) dq += (long)H[s][p] - (long)truth[s][p]; for (int p : small) dr += ((long)H[s][p] - (long)truth[s][p]) * psize(p);
              long d1 = 0; for (int p : small) if (psize(p) == 1) d1 += (long)H[s][p] - (long)truth[s][p];
              e1 += std::abs(dq); e2 += std::abs(dr); maxabs = std::max(maxabs, std::labs(d1));
              if (s % 4 == 1 && getenv("VERB") && (int)b == atoi(getenv("VERB"))) { printf("   seg %u: dQ %ld dR %ld d(1g) %ld | truth", s, dq, dr, d1); for (int p = 0; p < np; ++p) printf(" %u/%zu", truth[s][p], q[p].size()); printf(" | guess"); for (int p = 0; p < np; ++p) printf(" %u", H[s][p]); printf("\n"); } }
          printf("guess: busy %d, mean |dQ| %.2f, mean |dR| %.2f, max |d 1g| %ld\n", busy, e1 / busy, e2 / busy, maxabs); }
        // ---- rounds, absolute chaining (with optional warm-up: segment s re-simulates from the entry of the segment 'warm' GPUs earlier)
        std::vector<Heads> E(S + 1), Hn(S + 1);
        auto cq = [&](const Heads& h) { long c = 0; for (int p : big) c += h[p]; return c; };
        auto cr = [&](const Heads& h) { long c = 0; for (int p : small) c += (long)h[p] * psize(p); return c; };
        std::vector<double> lq(S, 1.0), lr(S, 1.0); std::vector<long> peq(S), pxq(S), per(S), pxr(S); std::vector<bool> have(S, false);
        // the pair of the small group (its longest single-slice and wider queue) and the hungry test of LEAD: the wider profile's pending request
        // is more than LEAD request-times older than the single-slice one's at both ends of the segment
        int pl = -1, ph = -1; for (int p : small) { if (psize(p) == 1 && (pl < 0 || q[p].size() > q[pl].size())) pl = p; if (psize(p) > 1 && (ph < 0 || q[p].size() > q[ph].size())) ph = p; }
        const long lead_th = getenv("LEAD") ? atol(getenv("LEAD")) : -1;
        auto lead = [&](const Heads& hh) { long t1 = hh[pl] < q[pl].size() ? (long)q[pl][hh[pl]] : (long)n, t2 = hh[ph] < q[ph].size() ? (long)q[ph][hh[ph]] : (long)n; return t1 - t2; };
        // EXPERT variants: DMASS=1 the Newton candidate's mass target is the sum of the masses the stages in front consumed (what the device
        // can compute from the D records) instead of this round's new entry of the stage in front; SCORE1=1 the candidates of round 1 are scored
        // too (the device before r03); LEADLAG=1 the pass-through uses the change of the exit in front since the previous round (observable
        // without a same-round prefix) instead of the change of its entry this round
        const bool dmass = getenv("DMASS") != nullptr, score1 = getenv("SCORE1") != nullptr, leadlag = getenv("LEADLAG") != nullptr;
        std::vector<Heads> Ep(S + 1, h0);
        const int secant = getenv("SECANT") ? atoi(getenv("SECANT")) : 0;
        std::vector<Heads> predA(S + 2), predB(S + 2); std::vector<bool> havePred(S + 2, false);
        std::vector<Heads> pH(S), pE(S); std::vector<bool> haveR(S, false); std::vector<double> lam(S, getenv("LAM0") ? atof(getenv("LAM0")) : 0.0);
        int rounds = 0; uint64_t crit = 0; uint32_t frontier = 0, frontier1 = 0, frontier2 = 0; uint64_t ncapped = 0;
        std::vector<Heads> Hsim(S), Xlast(S), Hc(S), Xc(S); std::vector<bool> logvalid(S, false), havec(S, false); std::vector<uint64_t> maxdec(S, 0);
        while (true) {
            ++rounds; uint64_t maxw = 0;
            uint32_t maxs = 0; uint64_t sumw = 0, nb_ = 0, second = 0;
            const bool docap = getenv("CAP") != nullptr; const double capf = docap ? atof(getenv("CAP")) : 0;
            for (uint32_t s = 0; s < S; ++s) {
                uint64_t d = 0;
                const bool resim = rounds == 1 || H[s] != Hsim[s] || !logvalid[s];
                if (!resim) { E[s + 1] = Xlast[s]; continue; }
                Heads ex = simulate(L.occ, s * seg, std::min(G, (s + 1) * seg), H[s], &d);
                const uint64_t cap = (uint64_t)(capf * maxdec[s]) + 64;
                const bool exempt = !docap || !havec[s] || s <= frontier2;
                if (!exempt && d > cap) {      // declined: extrapolate from the last complete simulation (what the successors would assume anyway)
                    d = cap; logvalid[s] = false; Hsim[s] = H[s];
                    long dq = 0, dr = 0; for (int p : big) dq += (long)H[s][p] - (long)Hc[s][p]; for (int p : small) dr += ((long)H[s][p] - (long)Hc[s][p]) * psize(p);
                    Heads h = Xc[s];
                    long nb = 0, ns = 0; for (int p : big) nb += q[p].size(); for (int p : small) ns += (long)q[p].size() * psize(p);
                    auto clampadd = [&](int p, long dd) { long v = (long)h[p] + dd; v = std::max(0l, std::min<long>(v, q[p].size())); h[p] = v; };
                    { std::vector<int> b2 = big; long dd = dq, tot = nb; std::sort(b2.begin(), b2.end());
                      for (size_t i = 0; i < b2.size(); ++i) { int p = b2[i]; long dp = i + 1 == b2.size() ? dd : (tot ? std::lround((double)dd * q[p].size() / tot) : 0); clampadd(p, dp); dd -= dp; tot -= q[p].size(); } }
                    { std::vector<int> grp = small; long dd = dr, tot = ns; std::sort(grp.begin(), grp.end(), [&](int x, int y) { return psize(x) > psize(y) || (psize(x) == psize(y) && x < y); });
                      for (size_t i = 0; i < grp.size(); ++i) { int p = grp[i]; long w = psize(p); long dp = i + 1 == grp.size() ? dd / w : (tot ? std::lround((double)dd * q[p].size() / tot) : 0); clampadd(p, dp); dd -= dp * w; tot -= (long)q[p].size() * w; } }
                    E[s + 1] = h; Xlast[s] = h; ++ncapped;
                } else {
                    E[s + 1] = ex; Xlast[s] = ex; Hsim[s] = H[s]; logvalid[s] = true; Hc[s] = H[s]; Xc[s] = ex; havec[s] = true; maxdec[s] = std::max<uint64_t>(maxdec[s], d);
                }
                if (d > maxw) { second = maxw; maxw = d; maxs = s; } else if (d > second) second = d; sumw += d; nb_ += d > 0;
            }
            if (getenv("VERBM") && (int)b == atoi(getenv("VERBM"))) printf("      round %d: max %lu at stage %u (second %lu), mean busy %.0f, frontier %u\n", rounds, maxw, maxs, second, nb_ ? (double)sumw / nb_ : 0.0, frontier);
            crit += maxw;
            Hn[0] = h0;
            auto hungry_at = [&](uint32_t s) { return lead_th >= 0 && pl >= 0 && ph >= 0 && lead(H[s]) > lead_th && lead(E[s + 1]) > lead_th; };
            std::vector<long> sumDq(S + 1, 0), sumDr(S + 1, 0);
            for (uint32_t s = 0; s < S; ++s) { sumDq[s + 1] = sumDq[s] + cq(E[s + 1]) - cq(H[s]); sumDr[s + 1] = sumDr[s] + cr(E[s + 1]) - cr(H[s]); }
            for (uint32_t s = 0; s < S; ++s) {
                Hn[s + 1] = E[s + 1];
                if (getenv("EXPERT") && rounds >= (score1 ? 1 : 2)) {
                    // candidates for stage s+1's next entry
                    Heads A = E[s + 1];
                    { long dq = 0, dr = 0; for (int p : big) dq += (long)Hn[s][p] - (long)H[s][p]; for (int p : small) dr += ((long)Hn[s][p] - (long)H[s][p]) * psize(p);
                      if (dmass) { dq = sumDq[s + 1] - cq(E[s + 1]); dr = sumDr[s + 1] - cr(E[s + 1]); }
                      long nb = 0, ns = 0; for (int p : big) nb += q[p].size(); for (int p : small) ns += (long)q[p].size() * psize(p);
                      auto clampadd = [&](int p, long d) { long v = (long)A[p] + d; v = std::max(0l, std::min<long>(v, q[p].size())); A[p] = v; };
                      { std::vector<int> b2 = big; long d = dq, tot = nb; std::sort(b2.begin(), b2.end()); for (size_t i = 0; i < b2.size(); ++i) { int p = b2[i]; long dp = i + 1 == b2.size() ? d : (tot ? std::lround((double)d * q[p].size() / tot) : 0); clampadd(p, dp); d -= dp; tot -= q[p].size(); } }
                      { std::vector<int> grp = small; long d = dr, tot = ns; std::sort(grp.begin(), grp.end(), [&](int x, int y) { return psize(x) > psize(y) || (psize(x) == psize(y) && x < y); });
                        for (size_t i = 0; i < grp.size(); ++i) { int p = grp[i]; long w = psize(p); long dp = i + 1 == grp.size() ? d / w : (tot ? std::lround((double)d * q[p].size() / tot) : 0); clampadd(p, dp); d -= dp * w; tot -= (long)q[p].size() * w; } } }
                    if (s > 0 && hungry_at(s)) {
                        // hungry stage in front: the split inside the small group passes through it, so its exit moves as its entry does
                        for (int p : small) { long sh = leadlag ? (long)E[s + 1][p] - (long)Ep[s + 1][p] : (long)Hn[s][p] - (long)H[s][p];
                            long v = (long)E[s + 1][p] + sh; A[p] = (uint32_t)std::max(0l, std::min<long>(v, q[p].size())); }
                    }
                    Heads Bc = E[s + 1];
                    // which rule would have predicted this round's entry better last round?  errA[s+1], errB[s+1] were recorded then
                    auto dist = [&](const Heads& x, const Heads& y) { long d = 0; for (int p = 0; p < np; ++p) d += std::labs((long)x[p] - (long)y[p]); return d; };
                    const long eA = !havePred[s + 1] ? 0 : dist(predA[s + 1], E[s + 1]), eB = !havePred[s + 1] ? 0 : dist(predB[s + 1], E[s + 1]);
                    // (the better predictor of the predecessor's exit as it turned out now)
                    predA[s + 1] = A; predB[s + 1] = Bc; havePred[s + 1] = true;
                    Hn[s + 1] = eB < eA ? Bc : A;
                    continue;
                }
                if (getenv("IDENT")) { for (int p = 0; p < np; ++p) { long v = (long)E[s + 1][p] + (long)Hn[s][p] - (long)H[s][p]; Hn[s + 1][p] = (uint32_t)std::max(0l, std::min<long>(v, q[p].size())); } continue; }
                if (!newton) continue;
                long dq = 0, dr = 0; for (int p : big) dq += (long)Hn[s][p] - (long)H[s][p]; for (int p : small) dr += ((long)Hn[s][p] - (long)H[s][p]) * psize(p);
                if (getenv("LQ")) { dq = std::lround(atof(getenv("LQ")) * dq); }
                if (getenv("LR")) { dr = std::lround(atof(getenv("LR")) * dr); }
                if (secant) {
                    const long eq = cq(H[s]), xq = cq(E[s + 1]), er = cr(H[s]), xr = cr(E[s + 1]);
                    if (have[s]) { if (eq != peq[s]) lq[s] = std::min(1.0, std::max(0.0, double(xq - pxq[s]) / double(eq - peq[s])));
                                   if (er != per[s]) lr[s] = std::min(1.0, std::max(0.0, double(xr - pxr[s]) / double(er - per[s]))); }
                    have[s] = true; peq[s] = eq; pxq[s] = xq; per[s] = er; pxr[s] = xr;
                    dq = std::lround(lq[s] * dq); dr = std::lround(lr[s] * dr);
                }
                Heads& h = Hn[s + 1];
                const Heads base_exit = E[s + 1];
                if (getenv("PROPA")) {
                    long nb = 0, ns = 0; for (int p : big) nb += q[p].size(); for (int p : small) ns += (long)q[p].size() * psize(p);
                    auto clampadd = [&](int p, long d) { long v = (long)h[p] + d; v = std::max(0l, std::min<long>(v, q[p].size())); h[p] = v; };
                    // exact in mass: the heaviest profiles first, the lightest one takes the remainder
                    auto spread = [&](std::vector<int> grp, long d, long tot) {
                        std::sort(grp.begin(), grp.end(), [&](int x, int y) { return psize(x) > psize(y) || (psize(x) == psize(y) && x < y); });
                        for (size_t i = 0; i < grp.size(); ++i) { int p = grp[i]; long w = psize(p);
                            long dp = i + 1 == grp.size() ? d / w : (tot ? std::lround((double)d * q[p].size() / tot) : 0);
                            clampadd(p, dp); d -= dp * w; tot -= (long)q[p].size() * w; }
                    };
                    { std::vector<int> b2 = big; long d = dq, tot = nb; std::sort(b2.begin(), b2.end());
                      for (size_t i = 0; i < b2.size(); ++i) { int p = b2[i]; long dp = i + 1 == b2.size() ? d : (tot ? std::lround((double)d * q[p].size() / tot) : 0); clampadd(p, dp); d -= dp; tot -= q[p].size(); } }
                    spread(small, dr, ns);
                    if (getenv("LEAD")) {
                        // hungry regime: the heavier small profile's pending request is much older than the lighter one's at both ends of the segment ->
                        // it takes every span it can use, the split inside the group passes through the segment unchanged
                        if (hungry_at(s)) { for (int p : small) { long v = (long)base_exit[p] + (long)Hn[s][p] - (long)H[s][p]; h[p] = (uint32_t)std::max(0l, std::min<long>(v, q[p].size())); } }
                    }
                    if (getenv("RESID")) {
                        // what the mass step did: m = h - base_exit; the entry shift was sh = Hn[s] - H[s]; residual r = sh - m (zero mass per group); pass lambda_s * r on
                        std::array<double, P> r{}; double nr = 0;
                        for (int p = 0; p < np; ++p) { r[p] = ((double)Hn[s][p] - (double)H[s][p]) - ((double)h[p] - (double)base_exit[p]); nr += r[p] * r[p]; }
                        // lambda estimate of stage s from its last two (entry, exit) pairs
                        if (haveR[s]) {
                            std::array<double, P> ri{}, ro{}; double a = 0, bb = 0;
                            // residuals of the entry change and of the exit change between the last two simulations (mass part removed with the same spread)
                            Heads z{}; 
                            auto massres = [&](const Heads& a1, const Heads& a0, std::array<double, P>& out) {
                                long mq = 0, mr = 0; for (int p : big) mq += (long)a1[p] - (long)a0[p]; for (int p : small) mr += ((long)a1[p] - (long)a0[p]) * psize(p);
                                Heads t = a0; Heads& hh = t;
                                auto clampadd2 = [&](int p, long d) { long v = (long)hh[p] + d; hh[p] = (uint32_t)std::max(0l, v); };
                                { std::vector<int> b2 = big; long d = mq, tot = nb; std::sort(b2.begin(), b2.end());
                                  for (size_t i = 0; i < b2.size(); ++i) { int p = b2[i]; long dp = i + 1 == b2.size() ? d : (tot ? std::lround((double)d * q[p].size() / tot) : 0); clampadd2(p, dp); d -= dp; tot -= q[p].size(); } }
                                { std::vector<int> grp = small; long d = mr, tot = ns; std::sort(grp.begin(), grp.end(), [&](int x, int y) { return psize(x) > psize(y) || (psize(x) == psize(y) && x < y); });
                                  for (size_t i = 0; i < grp.size(); ++i) { int p = grp[i]; long w = psize(p); long dp = i + 1 == grp.size() ? d / w : (tot ? std::lround((double)d * q[p].size() / tot) : 0); clampadd2(p, dp); d -= dp * w; tot -= (long)q[p].size() * w; } }
                                for (int p = 0; p < np; ++p) out[p] = ((double)a1[p] - (double)a0[p]) - ((double)t[p] - (double)a0[p]);
                            };
                            massres(H[s], pH[s], ri); massres(E[s + 1], pE[s], ro);
                            for (int p = 0; p < np; ++p) { a += ro[p] * ri[p]; bb += ri[p] * ri[p]; }
                            if (bb > 0) lam[s] = std::min(1.0, std::max(0.0, a / bb));
                        }
                        if (H[s] != pH[s] || !haveR[s]) { pH[s] = H[s]; pE[s] = E[s + 1]; haveR[s] = true; }
                        for (int p = 0; p < np; ++p) { long v = (long)h[p] + std::lround(lam[s] * r[p]); h[p] = (uint32_t)std::max(0l, std::min<long>(v, q[p].size())); }
                    }
                    continue;
                }
                // big group: advance / retreat |dq| requests in merged time order
                while (dq > 0) { int bp = -1; uint32_t bt = 0xFFFFFFFFu; for (int p : big) if (h[p] < q[p].size() && q[p][h[p]] < bt) { bt = q[p][h[p]]; bp = p; } if (bp < 0) break; ++h[bp]; --dq; }
                while (dq < 0) { int bp = -1; long bt = -1; for (int p : big) if (h[p] > 0 && (long)q[p][h[p] - 1] > bt) { bt = q[p][h[p] - 1]; bp = p; } if (bp < 0) break; --h[bp]; ++dq; }
                // small group: same rule weighted by size (advance the class whose next request is earliest)
                while (dr > 0) { int bp = -1; uint32_t bt = 0xFFFFFFFFu; for (int p : small) if (h[p] < q[p].size() && psize(p) <= dr && q[p][h[p]] < bt) { bt = q[p][h[p]]; bp = p; } if (bp < 0) break; ++h[bp]; dr -= psize(bp); }
                while (dr < 0) { int bp = -1; long bt = -1; for (int p : small) if (h[p] > 0 && psize(p) <= -dr && (long)q[p][h[p] - 1] > bt) { bt = q[p][h[p] - 1]; bp = p; } if (bp < 0) break; --h[bp]; dr += psize(bp); }
            }
            Ep = E;
            bool any = false; uint32_t wrong = 0;
            for (uint32_t s = 0; s <= S; ++s) { if (Hn[s] != H[s]) any = true; if (Hn[s] != truth[s]) ++wrong; H[s] = Hn[s]; }
            if (getenv("VERB") && (int)b == atoi(getenv("VERB"))) { printf("      err:"); for (uint32_t s = 0; s < 48 && s <= S; ++s) { long d = 0; for (int p = 0; p < np; ++p) d += std::labs((long)H[s][p] - (long)truth[s][p]); printf(" %ld", d); } printf("\n"); }
            if (getenv("VERBL") && (int)b == atoi(getenv("VERBL")) && rounds <= 16) { printf("      lam r%d:", rounds); for (uint32_t s = 0; s < 60; ++s) printf(" %.1f", lam[s]); printf("\n"); }
            if (getenv("VERBP") && (int)b == atoi(getenv("VERBP")) && rounds >= 12 && rounds <= 14) { for (uint32_t s = 24; s < 40; ++s) { printf("      r%d b%u:", rounds, s); for (int p = 0; p < np; ++p) printf(" %ld", (long)H[s][p] - (long)truth[s][p]); printf("\n"); } }
            frontier2 = frontier1; frontier1 = frontier;
            frontier = 0; while (frontier <= S && H[frontier] == truth[frontier]) ++frontier;
            printf("   round %d: boundaries still wrong %u, exact frontier %u / %u\n", rounds, wrong, frontier, S + 1);
            bool allvalid = true; for (uint32_t s = 0; s < S; ++s) if (!logvalid[s]) allvalid = false;
            if ((!any && allvalid) || rounds > 200) break;
        }
        printf("%s batch %zu seg %u: sequential decisions %lu | rounds %d, critical path %lu decisions (%.3fx) capped %lu\n", cfg.c_str(), b, seg, dec, rounds, crit, (double)crit / dec, ncapped);
        L.occ = occ_new; off += n;
    }
}
