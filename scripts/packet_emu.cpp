// packet_emu.cpp -- CPU emulation of the 64-query packet walk (pc_packet_traverse<2> + pc_scan_leaf_x2 of query_kernels.cuh)
// that COUNTS what a warp executes: node visits, leaf scans, and the fp64 re-checks of the leaf scans under two schemes:
//   per point  one fp64 block per point and query slot, entered when any lane's query passes d2 <= thr for that point
//              (the scan before the exact-leaf change: 2 x PC_LEAF sites per leaf)
//   per slot   pc_exact_leaf: one fp64 site per query slot, iterated once per point within the fp32 margin of the leaf's
//              minimum; the warp runs it as often as its busiest lane needs
// "warp" counts blocks the warp executes (any lane active), "lane" counts fp64 evaluations of single queries.
// Optionally the walk starts from an entry frontier instead of the root: the subtrees that meet the packet's bounding box
// dilated by `dil`, expanded breadth-first from the root while they number at most K (a grid "entry table" would store
// such frontiers per cell; the table lookup itself is not counted).
// Both schemes give the same result; with "check" every query is compared with an fp64 brute force (small inputs only).
// usage: packet_emu <points.bin> <queries.bin> <bound> [K=<entries>] [dil=<m>] [stride=<packets>] [check]
//        the queries are put into packets here, ordered by the top 24 bits of their Hilbert key in the index's frame;
//        bound = radius bound (max_radius + search_margin), 0 = unbounded (no entry frontier then)
#include <string>
#include "../tests/c/lbvh_host_build.hpp"

struct Packet {
    float q[64][3]; double best[64]; int32_t idx[64]; float thr[64]; int n;
};

struct Counts {
    int64_t packets = 0, visits = 0, leaf_scans = 0;
    int64_t warp_point = 0, lane_point = 0;      // fp64 blocks / evaluations, one site per point
    int64_t warp_slot = 0, lane_slot = 0;        // ... one site per query slot (pc_exact_leaf)
};

static inline double exact_d2(const pc_f4 &p, const float *q)
{
    const double ex = (double)p.x - (double)q[0], ey = (double)p.y - (double)q[1], ez = (double)p.z - (double)q[2];
    double e = ex * ex; e = e + ey * ey; e = e + ez * ez;
    return e;
}

// round-up fp32 of dmin * (1 + 2^-20) + 2^-147 (the __fmaf_ru of pc_exact_leaf, bounded from above by one ulp)
static inline float slot_cut(float dmin)
{
    const double c = (double)dmin * 1.00000095367431640625 + std::ldexp(1.0, -147);
    float f = (float)c;
    if ((double)f < c) f = nextafterf(f, INFINITY);
    return f;
}

static void scan_leaf(const LhIndex &ix, uint32_t ref, Packet &p, Counts &C)
{
    C.leaf_scans++;
    const pc_f4 *pt = ix.pts.data() + (ref & 0x7fffffffu);
    for (int j = 0; j < 2; j++) {                                 // query slot j of every lane: packet slots 32 j .. 32 j + 31
        bool point_block[PC_LBVH_LEAF] = {};
        int busiest = 0;
        for (int l = 0; l < 32; l++) {
            const int k = 32 * j + l;
            if (k >= p.n) break;
            float d[PC_LBVH_LEAF], dmin = FLT_MAX;
            for (int i = 0; i < PC_LBVH_LEAF; i++) {
                const float dx = pt[i].x - p.q[k][0], dy = pt[i].y - p.q[k][1], dz = pt[i].z - p.q[k][2];
                d[i] = std::fma(dz, dz, std::fma(dy, dy, dx * dx));
                dmin = std::min(dmin, d[i]);
            }
            if (!(dmin <= p.thr[k])) continue;
            // one site per point: the running threshold of the old scan, counted only
            float thr = p.thr[k]; double best = p.best[k]; int32_t idx = p.idx[k];
            for (int i = 0; i < PC_LBVH_LEAF; i++) {
                if (d[i] <= thr) {
                    point_block[i] = true; C.lane_point++;
                    const double e = exact_d2(pt[i], p.q[k]);
                    const int32_t id = (int32_t)pc_f2u(pt[i].w);
                    if (e < best || (e == best && (uint32_t)id < (uint32_t)idx)) { best = e; idx = id; thr = std::min(thr, lh_thr_from(e)); }
                }
            }
            // one site per slot: what the kernel does now, and what the walk continues with
            const float cut = std::min(p.thr[k], slot_cut(dmin));
            int cand = 0;
            for (int i = 0; i < PC_LBVH_LEAF; i++) {
                if (!(d[i] <= cut)) continue;
                cand++;
                const double e = exact_d2(pt[i], p.q[k]);
                const int32_t id = (int32_t)pc_f2u(pt[i].w);
                if (e < p.best[k] || (e == p.best[k] && (uint32_t)id < (uint32_t)p.idx[k])) { p.best[k] = e; p.idx[k] = id; }
            }
            p.thr[k] = std::min(p.thr[k], lh_thr_from(p.best[k]));
            if (p.best[k] != best || p.idx[k] != idx || p.thr[k] != thr) { fprintf(stderr, "the two leaf schemes disagree\n"); exit(3); }
            C.lane_slot += cand;
            busiest = std::max(busiest, cand);
        }
        for (int i = 0; i < PC_LBVH_LEAF; i++) C.warp_point += point_block[i];
        C.warp_slot += busiest;
    }
}

static inline float box_box_gap(const pc_f4 &mn, const pc_f4 &mx, const float *lo, const float *hi)
{
    const float g = std::max({ mn.x - hi[0], lo[0] - mx.x, mn.y - hi[1], lo[1] - mx.y, mn.z - hi[2], lo[2] - mx.z });
    return g;
}

static void walk(const LhIndex &ix, Packet &p, int K, float dil, Counts &C)
{
    uint32_t stack[256]; int sp = 0;
    if (ix.root & PC_REF_LEAF) { scan_leaf(ix, ix.root, p, C); return; }
    if (K <= 0) stack[sp++] = ix.root;
    else {
        // entry frontier: subtrees meeting the packet's box dilated by dil, at most K of them
        float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX }, c[3];
        for (int k = 0; k < p.n; k++) for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], p.q[k][a]); hi[a] = std::max(hi[a], p.q[k][a]); }
        for (int a = 0; a < 3; a++) { lo[a] -= dil; hi[a] += dil; c[a] = 0.5f * (lo[a] + hi[a]); }
        std::vector<uint32_t> F{ ix.root };
        for (bool grew = true; grew;) {                   // one level per pass
            grew = false;
            for (size_t at = 0; at < F.size();) {
                if (F[at] & PC_REF_LEAF) { at++; continue; }
                const pc_f4 *r = ix.rec.data() + 4 * (int64_t)F[at];
                std::vector<uint32_t> kids;
                for (int ch = 0; ch < 2; ch++)
                    if (box_box_gap(r[2 * ch], r[2 * ch + 1], lo, hi) <= 0.f) kids.push_back(pc_f2u(r[2 * ch].w));
                if ((int)(F.size() - 1 + kids.size()) > K) { at++; continue; }
                F.erase(F.begin() + (long)at);
                F.insert(F.begin() + (long)at, kids.begin(), kids.end());
                at += kids.size();
                grew = true;
            }
        }
        // leaves first, then the inner entries with the one nearest to the packet's centre on top of the stack
        std::vector<std::pair<float, uint32_t>> inner;
        for (uint32_t ref : F) {
            if (ref & PC_REF_LEAF) { scan_leaf(ix, ref, p, C); continue; }
            const pc_f4 *r = ix.rec.data() + 4 * (int64_t)ref;
            pc_f4 mn = r[0], mx = r[1];
            mn.x = std::min(mn.x, r[2].x); mn.y = std::min(mn.y, r[2].y); mn.z = std::min(mn.z, r[2].z);
            mx.x = std::max(mx.x, r[3].x); mx.y = std::max(mx.y, r[3].y); mx.z = std::max(mx.z, r[3].z);
            inner.push_back({ pc_lbvh_box_d2(mn, mx, c[0], c[1], c[2]), ref });
        }
        std::sort(inner.begin(), inner.end(), [](const std::pair<float, uint32_t> &a, const std::pair<float, uint32_t> &b) { return a.first > b.first; });
        for (auto &e : inner) stack[sp++] = e.second;
        if (sp == 0) return;
    }
    uint32_t ref = stack[--sp];
    for (;;) {
        C.visits++;
        const pc_f4 *r = ix.rec.data() + 4 * (int64_t)ref;
        float d0[64], d1[64];
        bool w0 = false, w1 = false;
        for (int k = 0; k < p.n; k++) {
            d0[k] = pc_lbvh_box_d2(r[0], r[1], p.q[k][0], p.q[k][1], p.q[k][2]);
            d1[k] = pc_lbvh_box_d2(r[2], r[3], p.q[k][0], p.q[k][1], p.q[k][2]);
            w0 = w0 || d0[k] <= p.thr[k]; w1 = w1 || d1[k] <= p.thr[k];
        }
        uint32_t next = 0xffffffffu;
        if (w0 || w1) {
            const bool both = w0 && w1;
            bool first0 = !w1;
            if (both) {                                   // vote of the lanes' first queries (slots 0..31) that are interested
                int interested = 0, pref0 = 0;
                for (int k = 0; k < std::min(p.n, 32); k++)
                    if (d0[k] <= p.thr[k] || d1[k] <= p.thr[k]) { interested++; if (d0[k] <= d1[k]) pref0++; }
                first0 = 2 * pref0 >= interested;
            }
            const uint32_t r0 = pc_f2u(r[0].w), r1 = pc_f2u(r[2].w);
            const uint32_t rn = first0 ? r0 : r1, rf = first0 ? r1 : r0;
            const float *dfar = first0 ? d1 : d0;
            if (rn & PC_REF_LEAF) scan_leaf(ix, rn, p, C); else next = rn;
            if (both) {
                if (rf & PC_REF_LEAF) {
                    bool still = false;                   // re-test against the bounds the near child may have tightened
                    for (int k = 0; k < p.n; k++) still = still || dfar[k] <= p.thr[k];
                    if (still) scan_leaf(ix, rf, p, C);
                } else if (next != 0xffffffffu) stack[sp++] = rf;
                else next = rf;
            }
        }
        if (next != 0xffffffffu) { ref = next; continue; }
        if (sp == 0) break;
        ref = stack[--sp];
    }
}

int main(int argc, char **argv)
{
    if (argc < 4) { fprintf(stderr, "usage: packet_emu <points.bin> <queries.bin> <bound> [K=n] [dil=m] [stride=n] [check]\n"); return 2; }
    int K = 0, stride = 1; float dil = 1.75f; bool check = false;
    for (int a = 4; a < argc; a++) {
        const std::string s = argv[a];
        if (s.rfind("K=", 0) == 0) K = atoi(s.c_str() + 2);
        else if (s.rfind("dil=", 0) == 0) dil = (float)atof(s.c_str() + 4);
        else if (s.rfind("stride=", 0) == 0) stride = std::max(1, atoi(s.c_str() + 7));
        else if (s == "check") check = true;
    }
    const std::vector<float> P = lh_read_f32(argv[1]);
    std::vector<float> Q = lh_read_f32(argv[2]);
    const double bound = atof(argv[3]);
    if (K > 0 && !(bound > 0 && bound <= dil)) { fprintf(stderr, "an entry frontier is exact only for bounded searches with bound <= dil\n"); return 2; }
    const int64_t m = (int64_t)Q.size() / 3;
    LhIndex ix;
    ix.build(P);
    std::vector<int64_t> ord((size_t)m); std::vector<uint32_t> key((size_t)m);
    for (int64_t k = 0; k < m; k++) { ord[(size_t)k] = k; key[(size_t)k] = ix.key_of(&Q[3 * k]) >> 6; }
    std::stable_sort(ord.begin(), ord.end(), [&](int64_t a, int64_t b) { return key[(size_t)a] < key[(size_t)b]; });
    float thr0 = FLT_MAX;
    if (bound > 0) {                                      // as pc_index.cu computes bound_thr
        const double b = bound * (1.0 + 1e-6), b2 = b * b * (1.0 + 1e-6);
        thr0 = nextafterf((float)b2, INFINITY) * 1.00000095367431640625f;
    }
    Counts C;
    int64_t bad = 0;
    for (int64_t base = 0; base < m; base += 64 * (int64_t)stride) {
        Packet p; p.n = (int)std::min<int64_t>(64, m - base);
        for (int k = 0; k < p.n; k++) { const int64_t s = ord[(size_t)(base + k)]; for (int a = 0; a < 3; a++) p.q[k][a] = Q[3 * s + a]; p.best[k] = INFINITY; p.idx[k] = -1; p.thr[k] = thr0; }
        C.packets++;
        if (ix.n > 0) walk(ix, p, K, dil, C);
        for (int k = 0; check && k < p.n; k++) {
            const int64_t s = ord[(size_t)(base + k)];
            double bb = INFINITY; int32_t bi = -1;
            for (int64_t i = 0; i < ix.n; i++) {
                const pc_f4 pi{ P[3 * i], P[3 * i + 1], P[3 * i + 2], 0.f };
                const double e = exact_d2(pi, &Q[3 * s]);
                if (e < bb) { bb = e; bi = (int32_t)i; }
            }
            const bool inside = bound <= 0 || bb <= (double)thr0;
            if (inside ? (bi != p.idx[k] || bb != p.best[k]) : (p.idx[k] != -1 && p.best[k] != bb)) { if (bad < 5) fprintf(stderr, "query %lld: got (%d, %.17g) want (%d, %.17g)\n", (long long)s, p.idx[k], p.best[k], bi, bb); bad++; }
        }
    }
    const double np = (double)std::max<int64_t>(C.packets, 1);
    printf("entries=%s n=%lld m=%lld packets=%lld visits/packet=%.1f leaf_scans/packet=%.1f fp64_warp/packet: per_point=%.1f per_slot=%.1f "
           "fp64_lane/packet: per_point=%.1f per_slot=%.1f mismatches=%s\n",
           K <= 0 ? "root" : ("K=" + std::to_string(K)).c_str(), (long long)ix.n, (long long)m, (long long)C.packets, C.visits / np, C.leaf_scans / np,
           C.warp_point / np, C.warp_slot / np, C.lane_point / np, C.lane_slot / np, check ? std::to_string(bad).c_str() : "unchecked");
    return bad ? 1 : 0;
}
