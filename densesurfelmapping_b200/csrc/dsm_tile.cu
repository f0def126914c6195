// Tile kernels of the superpixel pipeline (the default schedule): filtered assign pass, fused window-gather +
// Huber-Newton update on TMA-staged seed tiles, fused pixel-normal + plane-fit gather, and the plane-fit solver.
//
// Why they look the way they do (measured on the round-1 kernels, profiles/r1_final_*.csv):
//  * assign was bound by the float<->double conversion unit: the reference's cost expression (:364-387) crosses
//    the float/double boundary seven times per (pixel, candidate).  Only the ARGMIN of the costs reaches the
//    labels, so k_assign2 evaluates the costs in plain fp32 with a rigorous error bound (a filtered predicate,
//    as in exact computational geometry): if the two smallest costs are separated by more than the bound the
//    argmin is certain; otherwise (exact ties, near ties: ~1e-5 of real pixels) the pixel is re-evaluated with
//    the reference's exact mixed-precision expression.  Labels stay bit-identical by construction.
//  * the window gathers were bound by the L1 data pipe (six 16-byte global loads per lane over 8 image rows,
//    4x redundant label tests, bank-conflicting compaction stores) and each was followed by a separate per-seed
//    kernel reading the lists back from L2.  k_update / k_plane_gather stage one 8x4-seed tile (72x40 pixels)
//    with three TMA tensor copies, scan windows with lane = window row (16 consecutive pixels per lane,
//    conflict-free LDS.128), compact into shared memory and run the order-sensitive per-seed math from there.
// All citations ":NNN" refer to /root/reference/surfel_fusion/src/fusion_functions.cpp.
#include "dsm_exact.cuh"
#include <cuda_pipeline.h>

// -------------------------------------------------------------------------------------------
// mbarrier / TMA helpers (raw PTX; one elected thread arms the barrier and issues the tensor copies)
// -------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); // visible to the async proxy before the first copy
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded wait: a descriptor or byte-count mistake must trap, not hang the GPU (each try_wait blocks for a hardware time slice).
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity)
{
    unsigned ok = 0;
    for (unsigned spin = 0; !ok; spin++)
    {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(bar), "r"(parity)
                     : "memory");
        if (!ok && spin > (1u << 20)) __trap();
    }
}
__device__ __forceinline__ void tma_load_3d(unsigned dst, const CUtensorMap *map, int x, int y, int z, unsigned bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
                 "l"(reinterpret_cast<unsigned long long>(map)), "r"(bar), "r"(x), "r"(y), "r"(z)
                 : "memory");
}

// byte <-> bit masks of packed u8 planes
__device__ __forceinline__ unsigned zero_bytes_to_nibble(unsigned x)
{ // bit j of the result set iff byte j of x is zero (exact: no borrow tricks)
    unsigned t = (x & 0x7f7f7f7fu) + 0x7f7f7f7fu;
    t = ~(t | x | 0x7f7f7f7fu);                // 0x80 in every zero byte
    return ((t >> 7) * 0x00204081u >> 21) & 0xfu; // bits 0, 8, 16, 24 -> bits 21..24 of the product
}
// 4-bit mask -> 0xff per set bit
__device__ __forceinline__ unsigned nibble_to_bytes(unsigned n) { return (((n & 0xfu) * 0x00204081u) & 0x01010101u) * 0xffu; }

// -------------------------------------------------------------------------------------------
// K1  slic_assign (filtered) — update_pixels_kernel (:389-453) + calculate_cost (:364-387)
//
// Every pixel of the 8 x 8 block [8j+4, 8j+12) x [8k+4, 8k+12) has the same (at most) 2 x 2 candidate seeds: columns
// {j, j+1}, rows {k, k+1} (:413-422); the pixel at column 8j+4 sees only column j (:418-420), the pixel at row 8k+4
// only row k.  So a CTA (16 x 8 threads) covers one seed-row band, the pixel rows 8k+4 .. 8k+11 (the first band is
// rows -4 .. 3, clipped to the image), and a run of 128 columns starting at 128a - 4; a thread owns the 8 pixels
// 8j+4 .. 8j+11 of one row, all with the candidate columns {j, j+1}: "column 8j+4" is pixel 0 of every thread and
// "row 8k+4" is row 0 of every band.  After pdl_enter() 17 threads build the CTA's candidate table in shared memory from
// the band's 2 x 17 seeds (x/4, y/4, intensity, 1/mean_depth as hi + lo, mean_depth > 0); a thread then reads its
// 2 x 2 candidates with a few LDS.  The table holds the same fp32 values the cost expressions have always used.
// The reference walks the image in raster order and skips a pixel whose current seed is `stable` at that moment
// (:400); `stable` flips during the walk (:445/:450).  Here every seed carries a time stamp (tstable: -1 = unstable
// since the start of the pass, DSM_STABLE, or the raster index at which it became unstable); pixels of seeds
// unstable from the start commit at once, the others are deferred to the frame's relaxation (SURVEY.md H1).  How the
// winner of a pixel is found:
//   fast path   costs in fp32 (FMA allowed).  Against the reference's value c = fl24(..fl53(..)) the fp32 value c~
//               differs by at most 2^-20 (c~ + c) + 1e-12: squared distance and intensity term carry <= 3 roundings of
//               2^-24 each on either side; the depth term uses 1/mean_depth as hi + lo (error 2^-48 / mean_depth,
//               absolute floor 400 (2 |D| eta + eta^2) <= 1e-12 for 1/mean_depth <= 1024) and the EXACT per-pixel
//               inverse depth (invd plane, correctly rounded once by the first pass).  The test below uses
//               2^-18 (m1 + m2) + 1e-10, i.e. >= 4x slack.  If the smallest and second smallest fp32 cost are
//               separated by more than that, the reference's float comparison (:427, :432, strict '<') picks the
//               same candidate whatever the visiting order, and it is below the 1e6 start value (m1 < 9e5).
//   exact path  everything else (ties -- common on synthetic constant images --, near ties, all costs >= 9e5):
//               calc_cost, expression by expression as the reference, with the seeds read from global memory.
// The first pass also writes the inverse-depth plane the later passes read instead of the depth image.
// The last CTA of a frame to finish (ticket counter) runs the raster-order `stable` relaxation (relax_frame) for
// that frame, so the pass needs no separate one-CTA-per-frame launch.
// -------------------------------------------------------------------------------------------
#define A_EPS 3.814697265625e-06f // 2^-18
#define A_ALPHA 1e-10f
#define A_BIG 1e30f
#define ASG_TX 16             // threads per pixel row of an assign CTA (8 rows): 128 pixel columns
#define ASG_COLS (ASG_TX + 1) // seed columns of the CTA's candidate table

__device__ __forceinline__ void relax_frame(const DsmDev &d, int b, int tid, int nthreads)
{
    const int n = __ldcg(&d.nlist[b]);
    if (n > 0)
    {
        const size_t fo = (size_t)b * d.px_stride;
        int2 *list = d.list + fo;
        int32_t *labels = d.labels + fo;
        uint8_t *codes = d.code + fo;
        int32_t *t = d.tstable + (size_t)b * d.S;
        for (;;)
        {
            int changed = 0;
            for (int e = tid; e < n; e += nthreads)
            {
                const int2 en = __ldcg(&list[e]);
                if (en.x < 0) continue; // already evaluated
                const int owner = __ldcg(&labels[en.x]);
                if (__ldcg(&t[owner]) < en.x)
                {
                    const int win = en.y & 0x0fffffff; // entry: winner seed | winner's candidate code << 28
                    labels[en.x] = win;
                    codes[en.x] = (uint8_t)(en.y >> 28);
                    list[e].x = -1;
                    if (__ldcg(&t[win]) > en.x) atomicMin(&t[win], en.x);
                    changed = 1;
                }
            }
            if (!__syncthreads_or(changed)) break;
        }
    }
    if (tid == 0)
    {
        d.nlist[b] = 0; // the deferred-pixel list of this pass is consumed
        d.done[b] = 0;
    }
}

// label code of a pixel: which of its (at most) 2x2 candidate seeds it is labelled with, c = 2*ix + iy over the columns
// {xa, xa+1} and rows {ya, ya+1} defined below (the candidate set depends on the pixel position only, :413-422), or
// DSM_CODE_NONE for a pixel the reference would have left without any label (input domain, DESIGN.md 1.3).  The u8 code
// plane mirrors the int32 labels; the passes that only need "is this pixel a member of seed s" read it instead
// (1 byte per pixel, and the test is a byte compare with a pattern that depends on the window position only).
#define DSM_CODE_NONE 4
#define DSM_CODE_NONE4 0x04040404u

// seed index of candidate code c (sidx0 = seed index of candidate 0); a pixel without winner is labelled 0
__device__ __forceinline__ int seed_of_code(unsigned c, int sidx0, int spw)
{
    return c == DSM_CODE_NONE ? 0 : sidx0 + (int)(c & 1u) * spw + (int)(c >> 1);
}
__device__ __forceinline__ int4 labels_of_codes(unsigned w, int sidx0, int spw)
{
    return make_int4(seed_of_code(w & 0xffu, sidx0, spw), seed_of_code((w >> 8) & 0xffu, sidx0, spw),
                     seed_of_code((w >> 16) & 0xffu, sidx0, spw), seed_of_code(w >> 24, sidx0, spw));
}
// (:404-405) my_inv = (float)(1.0 / (double)depth) for depth > 0.01: 53 >= 2*24+2 bits, so the double rounding is
// innocuous and the correctly rounded float reciprocal is the same value (-ftz=false: subnormals included)
__device__ __forceinline__ float inv_depth(float z) { return z > F_0p01_LO ? __frcp_rn(z) : 0.0f; }

template <bool FIRST>
__global__ void __launch_bounds__(128, 8) k_assign2(const __grid_constant__ DsmDev d)
{
    pdl_enter();
    __shared__ float4 s_sd[2][ASG_COLS]; // seed rows ya, ya + 1: (x/4, or 1e18 for a missing seed; I; 1/md hi; lo)
    __shared__ float s_syq[2][ASG_COLS]; // y/4 of the same seeds
    __shared__ int s_md[ASG_COLS];       // bit r: the seed of row ya + r has mean_depth > 0 or is missing
    __shared__ int s_last;
    const int b = d.frame0 + blockIdx.z;
    const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * ASG_TX + tx, lane = tid & 31;
    const int ya = (int)blockIdx.y - 1;                       // candidate seed rows {ya, ya + 1}
    const int y = 8 * ya + 4 + ty;
    const int xa = ASG_TX * (int)blockIdx.x - 1 + tx;         // candidate seed columns {xa, xa + 1}
    const int x0 = 8 * xa + 4;                                // the thread's pixels x0 .. x0 + 7
    const bool row0 = ty == 0;                                // y = 8 ya + 4 sees only seed row ya (:421-422)
    const int spw = d.spw;
    const int sidx0 = ya * spw + xa;                          // seed index of candidate 0
    const size_t so = (size_t)b * d.S, fo = (size_t)b * d.px_stride;
    const int po = y * d.Wp + x0;                             // pixel offset within the frame (H * Wp < 2^31)
    // bit i: pixel x0 + i is inside the image.  Quad q (pixels x0 + 4q .. x0 + 4q + 3) is loaded and stored when its
    // first pixel is: x0 + 4q is 16-byte aligned for the float planes and 4-byte aligned for the byte planes.
    const int nx = min(d.W - x0, 8);
    const unsigned pm = (y >= 0 && y < d.H && nx > 0) ? ((1u << nx) - 1u) & (xa < 0 ? 0xf0u : 0xffu) : 0u;

    unsigned gw[2] = {0u, 0u}, ocw[2] = {0u, 0u}; // gray bytes; current labels as candidate codes (later passes)
    float iv[8];                                  // inverse depths
#pragma unroll
    for (int q = 0; q < 2; q++)
    {
        const bool ld = (pm >> (4 * q)) & 1u;
        const int o = po + 4 * q;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ld)
        {
            gw[q] = *reinterpret_cast<const unsigned *>(d.gray + fo + o);
            if (FIRST)
            {
                v = *reinterpret_cast<const float4 *>(d.depth + fo + o);
                v = make_float4(inv_depth(v.x), inv_depth(v.y), inv_depth(v.z), inv_depth(v.w));
                *reinterpret_cast<float4 *>(d.invd + fo + o) = v;
            }
            else
            {
                v = *reinterpret_cast<const float4 *>(d.invd + fo + o);
                ocw[q] = *reinterpret_cast<const unsigned *>(d.code + fo + o);
            }
        }
        iv[4 * q] = v.x, iv[4 * q + 1] = v.y, iv[4 * q + 2] = v.z, iv[4 * q + 3] = v.w;
    }

    // candidate table of the band: 2 seed rows x 17 seed columns, one thread per column
    if (tid < ASG_COLS)
    {
        const int j = xa - tx + tid;
        int md = 0;
#pragma unroll
        for (int r = 0; r < 2; r++)
        {
            const int sr = ya + r;
            const bool v = j >= 0 && j < spw && sr >= 0 && sr < d.sph;
            // Coordinates are pre-scaled by 1/4 (exact), so that dist/16 (:374) is ax'^2 + ay'^2.  A missing candidate
            // reads seed 0 and sits 1e18 away: its cost (~1e36, finite) is never the minimum and the filter arithmetic
            // stays NaN-free.
            const int li = v ? sr * spw + j : 0;
            const float4 s4 = d.seed[so + li];
            const float2 hl = d.seed_hl[so + li];
            s_sd[r][tid] = make_float4(v ? s4.x * 0.25f : 1e18f, s4.z, hl.x, hl.y);
            s_syq[r][tid] = s4.y * 0.25f;
            md |= (s4.w > 0.f || !v) ? 1 << r : 0;
        }
        s_md[tid] = md;
    }
    __syncthreads();

    unsigned wcw[2] = {DSM_CODE_NONE4, DSM_CODE_NONE4}; // winner of every pixel as a candidate code
    if (pm)
    {
        // candidate c = 2*ix + iy  -> (xa,ya) (xa,yb) (xb,ya) (xb,yb): dx outer, dy inner (:413-414).  Row 0 of the band
        // does not see row yb, pixel 0 not column xb: those candidates are pushed away like missing ones.
        const float4 c0 = s_sd[0][tx], c1 = s_sd[1][tx], c2 = s_sd[0][tx + 1], c3 = s_sd[1][tx + 1];
        const float sxq[4] = {c0.x, row0 ? 1e18f : c1.x, c2.x, row0 ? 1e18f : c3.x};
        const float sI[4] = {c0.y, c1.y, c2.y, c3.y}, shi[4] = {c0.z, c1.z, c2.z, c3.z}, slo[4] = {c0.w, c1.w, c2.w, c3.w};
        const float syq[4] = {s_syq[0][tx], s_syq[1][tx], s_syq[0][tx + 1], s_syq[1][tx + 1]};
        const float fyq = (float)y * 0.25f;
        float ayy[4];
#pragma unroll
        for (int c = 0; c < 4; c++)
        {
            const float ay = syq[c] - fyq;
            ayy[c] = ay * ay;
        }
        // every valid candidate seed has mean_depth > 0 (:378): over all 4 / over column xa only (pixel 0)
        const int mrow = row0 ? 2 : 0;
        const int mda = s_md[tx] | mrow, mdb = s_md[tx + 1] | mrow;
        const bool allmd = (mda & mdb) == 3, allmd0 = mda == 3;
        const float fxq0 = (float)x0 * 0.25f;
        unsigned wlo = 0u, whi = 0u, uncertain = 0u;
#pragma unroll
        for (int i = 0; i < 8; i++)
        {
            const float fxq = i == 0 ? fxq0 : fxq0 + 0.25f * (float)i; // = (float)(x0 + i) * 0.25f exactly
            const float pi = (float)((gw[i >> 2] >> (8 * (i & 3))) & 0xffu), pv = iv[i];
            // all_has_depth (:443): every valid candidate has a depth and so has the pixel -> costs with the depth term, else without
            const float w = (pv > 0.f && (i == 0 ? allmd0 : allmd)) ? 400.f : 0.f;
            float cost[4];
#pragma unroll
            for (int c = 0; c < 4; c++)
            {
                const float ax = ((i == 0 && (c >> 1)) ? 1e18f : sxq[c]) - fxq;
                const float n = fmaf(ax, ax, ayy[c]);
                const float idf = sI[c] - pi;
                const float cn = fmaf(idf * idf, 0.01f, n);
                const float t = (shi[c] - pv) + slo[c];
                cost[c] = fmaf(t * t, w, cn);
            }
            const float lo01 = fminf(cost[0], cost[1]), hi01 = fmaxf(cost[0], cost[1]);
            const float lo23 = fminf(cost[2], cost[3]), hi23 = fmaxf(cost[2], cost[3]);
            const float m1 = fminf(lo01, lo23);
            const float m2 = fminf(fminf(fmaxf(lo01, lo23), fminf(hi01, hi23)), A_BIG); // second smallest, kept finite
            // argmin as c = 2*ix + iy; it is used only when certain (the minimum is then unique)
            const unsigned wc = (lo23 == m1 ? 2u : 0u) | ((cost[1] == m1 || cost[3] == m1) ? 1u : 0u);
            if (i < 4) wlo |= wc << (8 * i);
            else whi |= wc << (8 * (i - 4));
            const bool certain = (m2 - m1 > A_EPS * (m2 + m1) + A_ALPHA) && (m1 < 9e5f);
            if (!certain) uncertain |= 1u << i;
        }
        uncertain &= pm;
        if (uncertain)
        { // exact path: the reference's expression, candidate order and strict '<' (first wins).  Each lane walks its OWN
          // flagged pixels, so a warp pays max-per-lane (usually one) exact evaluations, not one per pixel slot.
            SeedC sc[4];
            bool sv[4];
#pragma unroll
            for (int c = 0; c < 4; c++)
            {
                const int sx = xa + (c >> 1), sy = ya + (c & 1);
                sv[c] = sx >= 0 && sx < spw && sy >= 0 && sy < d.sph && !(row0 && (c & 1));
                const int li = sv[c] ? sy * spw + sx : 0;
                const float4 s4 = d.seed[so + li];
                sc[c].x = s4.x, sc[c].y = s4.y, sc[c].I = s4.z, sc[c].md = s4.w;
                sc[c].inv = d.inv_md[so + li]; // 1.0 / (double)mean_depth, only consumed when mean_depth > 0 (:378)
            }
            const float fy = (float)y;
            while (uncertain)
            {
                const int i = __ffs(uncertain) - 1;
                uncertain &= uncertain - 1;
                const float fx = (float)(x0 + i);
                const float my_i = (float)d.gray[fo + po + i];
                const float my_inv = FIRST ? inv_depth(d.depth[fo + po + i]) : d.invd[fo + po + i];
                const double my_inv_d = (double)my_inv;
                float min_d = 1e6f, min_nd = 1e6f;
                int idx_d = DSM_CODE_NONE, idx_nd = DSM_CODE_NONE; // the reference's -1 (:409-411)
                bool all_has_depth = true;
#pragma unroll
                for (int c = 0; c < 4; c++)
                {
                    const bool valid = sv[c] && !((c >> 1) && i == 0);
                    float cnd, cdd;
                    const bool has = calc_cost(sc[c], my_i, my_inv, my_inv_d, fx, fy, cnd, cdd);
                    cdd = valid ? cdd : __int_as_float(0x7f800000);
                    cnd = valid ? cnd : __int_as_float(0x7f800000);
                    all_has_depth &= has || !valid;
                    const bool bd = cdd < min_d, bn = cnd < min_nd;
                    min_d = bd ? cdd : min_d;
                    idx_d = bd ? c : idx_d;
                    min_nd = bn ? cnd : min_nd;
                    idx_nd = bn ? c : idx_nd;
                }
                const unsigned wv = (unsigned)(all_has_depth ? idx_d : idx_nd);
                const int sh = 8 * (i & 3);
                if (i < 4) wlo = (wlo & ~(0xffu << sh)) | (wv << sh);
                else whi = (whi & ~(0xffu << sh)) | (wv << sh);
            }
        }
        // pixels outside the image have no winner
        const unsigned bm0 = nibble_to_bytes(pm), bm1 = nibble_to_bytes(pm >> 4);
        wcw[0] = (wlo & bm0) | (DSM_CODE_NONE4 & ~bm0);
        wcw[1] = (whi & bm1) | (DSM_CODE_NONE4 & ~bm1);
    }

    if (FIRST)
    { // every label is 0 and seed 0 is unstable: everything commits (:400)
#pragma unroll
        for (int q = 0; q < 2; q++)
            if ((pm >> (4 * q)) & 1u)
            {
                *reinterpret_cast<int4 *>(d.labels + fo + po + 4 * q) = labels_of_codes(wcw[q], sidx0, spw);
                *reinterpret_cast<unsigned *>(d.code + fo + po + 4 * q) = wcw[q];
            }
        return;
    }

    // ---- iterations 2..: commit / defer (SURVEY.md H1).  Only a pixel whose winner differs from its label has anything
    // to do: with winner == label an evaluated pixel keeps its label and its stamp update min(t[label], idx) is a no-op
    // (the owner is unstable, t[label] < 0 <= idx), and a deferred one could change nothing in the relaxation either (if
    // the raster scan evaluates it, t[label] < idx, the label does not change and the stamp t[winner] = t[label] is
    // already below idx).  So the switching pixels are found first, from the packed codes, and the stamps are read for
    // those few only.  (A pixel without winner keeps its label; outside the image winner and label are both NONE.)
    unsigned sw = zero_bytes_to_nibble(~(__vcmpne4(wcw[0], ocw[0]) & __vcmpne4(wcw[0], DSM_CODE_NONE4))) |
                  (zero_bytes_to_nibble(~(__vcmpne4(wcw[1], ocw[1]) & __vcmpne4(wcw[1], DSM_CODE_NONE4))) << 4);
    const unsigned long long wc64 = wcw[0] | ((unsigned long long)wcw[1] << 32);
    unsigned deferred = 0;
    if (sw)
    {
        const int32_t *ts = d.tstable + so;
        const unsigned long long oc64 = ocw[0] | ((unsigned long long)ocw[1] << 32);
        unsigned long long cm = 0; // bytes of the pixels that commit
        while (sw)
        {
            const int i = __ffs(sw) - 1;
            sw &= sw - 1;
            const int win = seed_of_code((unsigned)(wc64 >> (8 * i)) & 0xffu, sidx0, spw);
            if (ts[seed_of_code((unsigned)(oc64 >> (8 * i)) & 0xffu, sidx0, spw)] < 0)
            { // owner unstable since the start of the pass: the reference evaluates this pixel
                cm |= 0xffull << (8 * i);
                if (ts[win] > po + i) atomicMin(&d.tstable[so + win], po + i); // stable = false at time pidx (:445/:450)
            }
            else
                deferred |= 1u << i;
        }
        const unsigned long long nc = (oc64 & ~cm) | (wc64 & cm);
#pragma unroll
        for (int q = 0; q < 2; q++)
            if ((unsigned)(cm >> (32 * q)))
            {
                const unsigned w = (unsigned)(nc >> (32 * q));
                *reinterpret_cast<int4 *>(d.labels + fo + po + 4 * q) = labels_of_codes(w, sidx0, spw);
                *reinterpret_cast<unsigned *>(d.code + fo + po + 4 * q) = w;
            }
    }
    // warp-aggregated append of the deferred pixels (rare: most warps have none)
    const int nent = __popc(deferred);
    if (__any_sync(FULL, nent > 0))
    {
        int total;
        const int excl = warp_excl_scan(nent, lane, total);
        int base = 0;
        if (lane == 31) base = atomicAdd(&d.nlist[b], total);
        base = __shfl_sync(FULL, base, 31);
        int2 *list = d.list + fo + base + excl;
        while (deferred)
        {
            const int i = __ffs(deferred) - 1;
            deferred &= deferred - 1;
            const unsigned c = (unsigned)(wc64 >> (8 * i)) & 0xffu;
            *list++ = make_int2(po + i, seed_of_code(c, sidx0, spw) | (int)(c << 28)); // (pitched raster index, winner | code << 28)
        }
    }
    // frame-completion ticket: the CTA that takes the last ticket of frame b sees every other CTA's labels, list
    // entries and time stamps (release: fence before the ticket; acquire: fence after it) and resolves the frame
    __syncthreads(); // the CTA's writes happen-before thread 0's fence (fences are cumulative): one fence per CTA, as in a grid barrier
    if (tid == 0)
    {
        __threadfence();
        s_last = (atomicAdd(&d.done[b], 1) == (int)(gridDim.x * gridDim.y) - 1) ? 1 : 0;
    }
    __syncthreads();
    if (s_last)
    {
        __threadfence();
        relax_frame(d, b, tid, ASG_TX * 8);
    }
}

// -------------------------------------------------------------------------------------------
// K2  slic_update — update_seeds_kernel (:468-562), as a tile gather and a per-seed solve
//
// K2a k_gather (CTA = DSM_TILE_SX x DSM_TILE_SY = 32 seeds).  One thread arms an mbarrier and issues three TMA tensor
//   copies (labels, depth boxes of 76x41 elements at pixel (64 bx - 4, 32 by - 4), gray box of 112x41 at (64 bx - 16,
//   32 by - 4); out-of-image parts are zero-filled by the hardware and masked by coordinates below exactly like the
//   reference's clamped loops).  A half-warp serves one seed, lane = window row: a lane reads its row's 16 pixels with
//   conflict-free 16-byte shared loads and turns them into a 16-bit membership mask; count, sum x, sum y and sum
//   intensity (exactly representable integers < 2^24, so the reference's float accumulation is exact and order-free)
//   come from population counts and byte dot products of the mask and are combined over the 16 lanes by packed
//   xor-butterflies.  Member depths > 0.1 are compacted IN RASTER ORDER (row-major = lane order, then column order
//   inside the lane) into a per-seed list staged in shared memory and copied out as contiguous 16-byte runs:
//   dlist[b][seed][DL_STRIDE].
// K2b k_newton2 (thread per seed, every seed of the batch in flight): the float sums sum_depth (:511) and sum_a
//   (:536-549) feed the next pass's costs and are order-sensitive (SURVEY.md H2), so one thread walks its seed's list
//   sequentially, 8 entries (two 16-byte loads = one 32-byte sector) per step.  residual = fl(md - z) is monotone
//   in z, so the list's extremes (found during the mean pass) decide for ALL entries whether they are inside the
//   Huber range; in that -- by far most common -- case a Newton pass is a pure dependent chain
//   sum_a = fmaf(2, md - z, sum_a) (2 r is exact: the same single rounding as `sum_a += 2 * residual`).
// -------------------------------------------------------------------------------------------
#define DL_STRIDE 232 // floats per seed list: >= 15*15 possible members, multiple of 8 (32-byte sectors)
#define TILE_PLANE_BYTES 12544 // 76 * 41 * 4 = 12464 rounded up to 128: TMA destinations are 128-byte aligned
#define TILE_BYTE_PLANE 4608 // 112 * 41 = 4592 rounded up to 128
#define GAT_SMEM_DEP 0
#define GAT_SMEM_COD TILE_PLANE_BYTES
#define GAT_SMEM_GRY (TILE_PLANE_BYTES + TILE_BYTE_PLANE)
#define GAT_SMEM_LIST (TILE_PLANE_BYTES + 2 * TILE_BYTE_PLANE) // float [16][DL_STRIDE]: the 16 seeds of one round
#define GAT_SMEM_ND (GAT_SMEM_LIST + 16 * DL_STRIDE * 4)        // int [16] list lengths of the round
#define GAT_SMEM_BAR (GAT_SMEM_ND + 16 * 4)
#define GAT_SMEM_BYTES (GAT_SMEM_BAR + 16)
#define TILE_TX_BYTES (DSM_TILE_W * DSM_TILE_H * 4u + 2u * DSM_TILE_GW * DSM_TILE_H)

// 16-bit membership mask of one window row from the label-code tile: bit k set iff the pixel at window column k is labelled
// with the seed whose window this is.  Inside the 16 x 16 window of seed (sx, sy) the pixel at column k, row r sees that
// seed as candidate ix = (k < 8), iy = (r < 8) (its candidate columns are {sx-1, sx} for k < 8 and {sx, sx+1} otherwise,
// :413-422), i.e. the expected code byte is (k < 8 ? 2 : 0) | (r < 8 ? 1 : 0).  Four 32-bit words = 16 code bytes.
__device__ __forceinline__ unsigned member_mask16(const unsigned *codes, int r)
{
    const unsigned lo = (r < 8) ? 0x01010101u : 0u; // iy
    const unsigned e_left = 0x02020202u | lo, e_right = lo;
    return zero_bytes_to_nibble(codes[0] ^ e_left) | (zero_bytes_to_nibble(codes[1] ^ e_left) << 4) |
           (zero_bytes_to_nibble(codes[2] ^ e_right) << 8) | (zero_bytes_to_nibble(codes[3] ^ e_right) << 12);
}

// sum over the set bits k of a 16-bit mask of k: sum_j 2^j popc(mask & {k : bit j of k set})
__device__ __forceinline__ int mask_index_sum(unsigned m)
{
    return __popc(m & 0xaaaau) + 2 * __popc(m & 0xccccu) + 4 * __popc(m & 0xf0f0u) + 8 * __popc(m & 0xff00u);
}

__global__ void __launch_bounds__(256, 6) k_gather(const __grid_constant__ DsmDev d, const __grid_constant__ DsmMaps mp)
{
    pdl_enter();
    extern __shared__ __align__(128) unsigned char smem[];
    const float *t_dep = reinterpret_cast<const float *>(smem + GAT_SMEM_DEP);
    const uint8_t *t_cod = smem + GAT_SMEM_COD, *t_gry = smem + GAT_SMEM_GRY;
    float *lists = reinterpret_cast<float *>(smem + GAT_SMEM_LIST);
    int *s_nd = reinterpret_cast<int *>(smem + GAT_SMEM_ND);
    const unsigned bar = smem_u32(smem + GAT_SMEM_BAR);

    const int b = d.frame0 + blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int X0 = blockIdx.x * (DSM_TILE_SX * DSM_SP) - DSM_SP / 2, Y0 = blockIdx.y * (DSM_TILE_SY * DSM_SP) - DSM_SP / 2;
    if (threadIdx.x == 0)
    {
        mbar_init(bar, 1);
        mbar_expect_tx(bar, TILE_TX_BYTES);
        tma_load_3d(smem_u32(smem + GAT_SMEM_DEP), &mp.dep, X0, Y0, b, bar);
        tma_load_3d(smem_u32(smem + GAT_SMEM_COD), &mp.cod, X0 - DSM_TILE_GX, Y0, b, bar);
        tma_load_3d(smem_u32(smem + GAT_SMEM_GRY), &mp.gry, X0 - DSM_TILE_GX, Y0, b, bar);
    }
    if (threadIdx.x == 1 && blockIdx.x == 0 && blockIdx.y == 0) d.nhard[b] = 0; // this pass's queue of hard Newton seeds
    const int W = d.W, H = d.H;
    const size_t so = (size_t)b * d.S;
    const int half = lane >> 4, r = lane & 15;
    // the stable flags are fetched while the tile is in flight; stable seeds are skipped by update_seeds (:478-479)
    int tflag[2];
#pragma unroll
    for (int rd = 0; rd < 2; rd++)
    {
        const int sl = rd * 16 + warp * 2 + half;
        const int sp_x = blockIdx.x * DSM_TILE_SX + (sl & 7), sp_y = blockIdx.y * DSM_TILE_SY + (sl >> 3);
        const bool live = sp_x < d.spw && sp_y < d.sph;
        tflag[rd] = live ? d.tstable[so + sp_y * d.spw + sp_x] : DSM_STABLE;
    }
    __syncthreads(); // barrier initialised before anybody polls it
    mbar_wait(bar, 0);
#pragma unroll
    for (int rd = 0; rd < 2; rd++)
    {
        const int q = warp * 2 + half; // seed slot of this round
        const int sl = rd * 16 + q;
        const int tx = sl & 7, ty = sl >> 3;
        const int sp_x = blockIdx.x * DSM_TILE_SX + tx, sp_y = blockIdx.y * DSM_TILE_SY + ty;
        const int s = sp_y * d.spw + sp_x;
        const bool act = tflag[rd] != DSM_STABLE;
        const int x0 = sp_x * DSM_SP - DSM_SP / 2, y0 = sp_y * DSM_SP - DSM_SP / 2;
        const int xb = x0 > 0 ? x0 : 0, yb = y0 > 0 ? y0 : 0;
        const int xe = (x0 + 16) < W - 1 ? (x0 + 16) : W - 1; // end-exclusive: last row/col never visited (:488-489)
        const int ye = (y0 + 16) < H - 1 ? (y0 + 16) : H - 1;
        const int y = y0 + r;
        const bool rowin = act && y >= yb && y < ye;
        // member columns of the window: xb - x0 <= k < xe - x0; nothing if the row is outside
        const unsigned kmask = rowin ? (((1u << (xe - x0)) - 1u) & ~((1u << (xb - x0)) - 1u)) : 0u;
        const int trow = ty * DSM_SP + r, tcol = tx * DSM_SP;
        float zk[16];
        unsigned mm, zm = 0; // bit k: labelled with this seed / depth > 0.1
        {
            const unsigned *pc = reinterpret_cast<const unsigned *>(t_cod + trow * DSM_TILE_GW + DSM_TILE_GX + tcol); // 4-byte aligned
            const unsigned cw[4] = {pc[0], pc[1], pc[2], pc[3]};
            mm = member_mask16(cw, r);
            const float4 *pz = reinterpret_cast<const float4 *>(t_dep + trow * DSM_TILE_W + tcol);
#pragma unroll
            for (int qd = 0; qd < 4; qd++)
            {
                const float4 z = pz[qd];
                zk[4 * qd] = z.x, zk[4 * qd + 1] = z.y, zk[4 * qd + 2] = z.z, zk[4 * qd + 3] = z.w;
            }
#pragma unroll
            for (int k = 0; k < 16; k++) zm |= (zk[k] > F_0p1_LO ? 1u : 0u) << k; // (double)depth > 0.1 (:508)
        }
        mm &= kmask;
        const unsigned dm = mm & zm; // member with depth > 0.1
        const int cnt = __popc(mm);
        const int sdx = mask_index_sum(mm);
        int si = 0;
        {
            const unsigned *pg = reinterpret_cast<const unsigned *>(t_gry + trow * DSM_TILE_GW + DSM_TILE_GX + tcol); // 4-byte aligned
#pragma unroll
            for (int qd = 0; qd < 4; qd++) si = (int)__dp4a(pg[qd] & nibble_to_bytes(mm >> (4 * qd)), 0x01010101u, (unsigned)si);
        }
        // packed 16-lane butterflies: count <= 225 (8 bits) | sum intensity <= 57375 (16 bits);
        // sum (x - x0) <= 3375 (12 bits) | sum (y - y0) <= 3375
        int pa = cnt | (si << 8), pb = sdx | ((cnt * r) << 12);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1)
        {
            pa += __shfl_xor_sync(FULL, pa, o);
            pb += __shfl_xor_sync(FULL, pb, o);
        }
        const int c = __popc(dm);
        int incl = c;
#pragma unroll
        for (int o = 1; o < 16; o <<= 1)
        {
            const int nb = __shfl_up_sync(FULL, incl, o, 16);
            if (r >= o) incl += nb;
        }
        const int ndt = __shfl_sync(FULL, incl, 15, 16);
        if (rd) __syncthreads(); // the previous round's lists have been copied out
        float *lp = lists + q * DL_STRIDE + (incl - c);
#pragma unroll
        for (int k = 0; k < 16; k++)
            if ((dm >> k) & 1u) *lp++ = zk[k];
        if (r == 0)
        {
            s_nd[q] = act ? ndt : 0;
            if (act)
            {
                const int n = pa & 0xff;
                d.usum[so + s] = make_int4(n, n * x0 + (pb & 0xfff), n * y0 + (pb >> 12), pa >> 8);
                d.und[so + s] = ndt;
            }
        }
        __syncthreads();
        // copy-out: warp w moves the lists of seed slots w and w + 8 of this round -> dlist[b][seed][0 .. nd), 16 bytes per lane
#pragma unroll
        for (int h2 = 0; h2 < 2; h2++)
        {
            const int q2 = warp + 8 * h2, n2 = s_nd[q2];
            if (n2 == 0) continue; // warp-uniform
            const int sl2 = rd * 16 + q2;
            const int s2 = (blockIdx.y * DSM_TILE_SY + (sl2 >> 3)) * d.spw + blockIdx.x * DSM_TILE_SX + (sl2 & 7);
            float4 *dst = reinterpret_cast<float4 *>(d.dlist + (so + s2) * DL_STRIDE);
            const float4 *src = reinterpret_cast<const float4 *>(lists + q2 * DL_STRIDE);
            if (4 * lane < n2) dst[lane] = src[lane];
            if (4 * (lane + 32) < n2) dst[lane + 32] = src[lane + 32];
        }
    }
}

#define NW_T 64       // seeds (threads) per CTA of the two Newton kernels
#define NW_CAP 5632   // floats of list staging per CTA (22 KB): 88 entries per seed on average, 225 possible; 8 CTAs per SM
__global__ void __launch_bounds__(NW_T, 8) k_newton2(const __grid_constant__ DsmDev d)
{
    pdl_enter();
    // Every thread stages its seed's list (a contiguous run in global memory) into shared memory with 16-byte cp.async and
    // then walks it there up to six times.  Lists that do not fit (rare: NW_CAP covers 88 entries per seed) stay in global memory.
    __shared__ __align__(16) float buf[NW_CAP];
    __shared__ int s_off[NW_T], s_wsum[NW_T / 32];
    const int b = d.frame0 + blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = blockIdx.x * NW_T + tid;
    const size_t so = (size_t)b * d.S;
    // the four per-seed loads are independent and issued together (one memory round trip), before the list staging
    const bool inr = s < d.S;
    const int tflag = inr ? d.tstable[so + s] : DSM_STABLE;
    const int nd_raw = inr ? d.und[so + s] : 0;
    const int4 su = inr ? d.usum[so + s] : make_int4(0, 0, 0, 0);
    const float4 pre = inr ? d.seed[so + s] : make_float4(0.f, 0.f, 0.f, 0.f);
    const bool act = tflag != DSM_STABLE; // stable seeds are untouched by update_seeds (:478-479)
    const int nd = act ? nd_raw : 0;
    {
        const int len4 = (nd + 3) & ~3;
        int wtot;
        const int wex = warp_excl_scan(len4, lane, wtot);
        if (lane == 31) s_wsum[warp] = wtot;
        __syncthreads();
        int base = 0;
        for (int w = 0; w < warp; w++) base += s_wsum[w];
        const int off = base + wex;
        s_off[tid] = (off + len4 <= NW_CAP) ? off : -1;
    }
    // every thread copies its own list (a contiguous run in global memory) with 16-byte cp.async: all copies of the CTA are in
    // flight at once, no register staging, and a thread waits for its own copies only (it never reads another list)
    if (s_off[tid] >= 0)
    {
        const float4 *src = reinterpret_cast<const float4 *>(d.dlist + (so + s) * DL_STRIDE);
        float4 *dst = reinterpret_cast<float4 *>(buf + s_off[tid]);
        for (int j4 = 0; 4 * j4 < nd; j4++) __pipeline_memcpy_async(dst + j4, src + j4, 16);
    }
    __pipeline_commit();
    __pipeline_wait_prior(0);
    if (!act) return;
    // Every seed runs its mean pass and its Newton passes as long as every entry is inside the Huber range (a pure
    // dependent chain).  A seed that meets an out-of-range entry is appended to the frame's queue of hard seeds with its
    // state; k_newton_hard continues those, one thread each at full occupancy, so that the entry-by-entry
    // classification loop is never executed by a warp in which one lane needs it and 31 wait.
    if (act)
    {
        const int n = su.x;
        if (n == 0)
        { // unreachable for supported shapes (every seed keeps its centre pixel, SURVEY H3); recorded, never silently ignored
            atomicAdd(&d.errflag[b], 1);
            d.tstable[so + s] = -1;
        }
        else
        {
            const float fn = (float)n; // sums below are < 2^24 so the reference's float accumulation is exact
            const float mi = (float)su.w / fn;
            const float mx = (float)su.y / fn;
            const float my = (float)su.z / fn;
            // ::fabs(double): float differences, summed in double, rounded once (:527)
            const float diff = (float)(fabs((double)(pre.z - mi)) + fabs((double)(pre.x - mx)) + fabs((double)(pre.y - my)));
            const bool newstable = diff < F_0p2_HI; // (double)diff < 0.2 (:528)
            float md = 0.0f;
            bool queued = false;
            if (nd > 0)
            {
                const float *dl = s_off[tid] >= 0 ? buf + s_off[tid] : d.dlist + (so + s) * DL_STRIDE; // generic: shared or global
                const float4 *dl4 = reinterpret_cast<const float4 *>(dl);
                float sum_d = 0.0f, zmn = __int_as_float(0x7f800000), zmx = 0.f;
                {
                    int k = 0;
                    for (; k + 8 <= nd; k += 8)
                    {
                        const float4 a = dl4[k >> 2], c = dl4[(k >> 2) + 1];
                        const float v[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
#pragma unroll
                        for (int j = 0; j < 8; j++) sum_d += v[j]; // raster order (:511)
                        zmn = fminf(zmn, fminf(fminf(fminf(v[0], v[1]), fminf(v[2], v[3])), fminf(fminf(v[4], v[5]), fminf(v[6], v[7]))));
                        zmx = fmaxf(zmx, fmaxf(fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3])), fmaxf(fmaxf(v[4], v[5]), fmaxf(v[6], v[7]))));
                    }
                    for (; k < nd; k++)
                    {
                        const float v = dl[k];
                        sum_d += v;
                        zmn = fminf(zmn, v);
                        zmx = fmaxf(zmx, v);
                    }
                }
                md = sum_d / (float)nd;
                for (int it = 0; it < 5; it++)
                { // damped Huber-Newton (:534-554)
                    // residual = fl(md - z) is monotone in z: the list's extremes decide for ALL entries whether they are inside
                    // the Huber range ((double)r < HUBER_RANGE && (double)r > -HUBER_RANGE, :540)
                    if (!((md - zmn) < d.huber_hi && (md - zmx) > -d.huber_hi))
                    {
                        queued = true;
                        d.pfsum[(so + s) * 2] = make_float4(md, __int_as_float(it), zmn, zmx); // the plane-fit scratch is free during the clustering
                        break;
                    }
                    // every entry in range: sum_a += 2 * residual (2 r is exact, one rounding per add = fmaf(2, r, sum_a)),
                    // sum_b = nd exact additions of 2
                    float sa = 0.0f;
                    int k = 0;
                    for (; k + 8 <= nd; k += 8)
                    {
                        const float4 a = dl4[k >> 2], c = dl4[(k >> 2) + 1];
                        sa = fmaf(2.0f, md - a.x, sa), sa = fmaf(2.0f, md - a.y, sa), sa = fmaf(2.0f, md - a.z, sa), sa = fmaf(2.0f, md - a.w, sa);
                        sa = fmaf(2.0f, md - c.x, sa), sa = fmaf(2.0f, md - c.y, sa), sa = fmaf(2.0f, md - c.z, sa), sa = fmaf(2.0f, md - c.w, sa);
                    }
                    for (; k < nd; k++) sa = fmaf(2.0f, md - dl[k], sa);
                    const float delta = (float)((double)(-sa) / ((double)(float)(2 * nd) + 10.0));
                    md = md + delta;
                    if (delta < F_0p01_HI && delta > -F_0p01_HI) break; // |delta| < 0.01 in double (:552)
                }
            }
            if (queued)
            {
                d.pfsum[(so + s) * 2 + 1] = make_float4(mx, my, mi, newstable ? 1.f : 0.f);
                d.hardq[so + atomicAdd(&d.nhard[b], 1)] = s;
            }
            else
            {
                d.seed[so + s] = make_float4(mx, my, mi, md);
                d.seed_hl[so + s] = split_inverse(md);
                d.inv_md[so + s] = 1.0 / (double)md; // exact-path operand of the assign pass, only consumed when md > 0 (:378)
                d.tstable[so + s] = newstable ? DSM_STABLE : -1;
            }
        }
    }
}

// K2c k_newton_hard (thread per queued seed): the Newton passes of the seeds that have entries outside the Huber range
// (:540-547), continued from the state k_newton2 left.  Eight entries per step: their residuals and in-range flags are
// independent and computed first; what remains serial is the reference's running sum -- fmaf(2, r, sum_a) for an entry
// in range, (float)((double)sum_a + -+HUBER_RANGE) for one outside (:547).
__global__ void __launch_bounds__(NW_T, 8) k_newton_hard(const __grid_constant__ DsmDev d)
{
    pdl_enter();
    __shared__ __align__(16) float buf[NW_CAP];
    __shared__ int s_off[NW_T], s_wsum[NW_T / 32];
    const int b = d.frame0 + blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nq = d.nhard[b];
    if (blockIdx.x * NW_T >= nq) return; // whole CTA beyond the queue
    const int q = blockIdx.x * NW_T + tid;
    const size_t so = (size_t)b * d.S;
    const bool act = q < nq;
    const int s = act ? d.hardq[so + q] : 0;
    const int nd = act ? d.und[so + s] : 0;
    { // stage the CTA's lists into shared memory exactly like k_newton2 (coalesced cp.async, all in flight at once)
        const int len4 = (nd + 3) & ~3;
        int wtot;
        const int wex = warp_excl_scan(len4, lane, wtot);
        if (lane == 31) s_wsum[warp] = wtot;
        __syncthreads();
        int base = 0;
        for (int w = 0; w < warp; w++) base += s_wsum[w];
        const int off = base + wex;
        s_off[tid] = (off + len4 <= NW_CAP) ? off : -1;
    }
    if (s_off[tid] >= 0)
    {
        const float4 *src = reinterpret_cast<const float4 *>(d.dlist + (so + s) * DL_STRIDE);
        float4 *dst = reinterpret_cast<float4 *>(buf + s_off[tid]);
        for (int j4 = 0; 4 * j4 < nd; j4++) __pipeline_memcpy_async(dst + j4, src + j4, 16);
    }
    __pipeline_commit();
    const float4 st = d.pfsum[(so + s) * 2], mn = d.pfsum[(so + s) * 2 + 1]; // in flight together with the list copies
    __pipeline_wait_prior(0);
    if (!act) return;
    const float *dl = s_off[tid] >= 0 ? buf + s_off[tid] : d.dlist + (so + s) * DL_STRIDE; // generic: shared or global
    const float4 *dl4 = reinterpret_cast<const float4 *>(dl);
    float md = st.x;
    const float zmn = st.z, zmx = st.w;
    const double hp = d.huber, hm = -1 * d.huber;
    for (int it = __float_as_int(st.y); it < 5; it++)
    {
        float sa = 0.0f, sb = 0.0f;
        if ((md - zmn) < d.huber_hi && (md - zmx) > -d.huber_hi)
        { // back inside the range with every entry: the pure chain
            int k = 0;
            for (; k + 8 <= nd; k += 8)
            {
                const float4 a = dl4[k >> 2], c = dl4[(k >> 2) + 1];
                sa = fmaf(2.0f, md - a.x, sa), sa = fmaf(2.0f, md - a.y, sa), sa = fmaf(2.0f, md - a.z, sa), sa = fmaf(2.0f, md - a.w, sa);
                sa = fmaf(2.0f, md - c.x, sa), sa = fmaf(2.0f, md - c.y, sa), sa = fmaf(2.0f, md - c.z, sa), sa = fmaf(2.0f, md - c.w, sa);
            }
            for (; k < nd; k++) sa = fmaf(2.0f, md - dl[k], sa);
            sb = (float)(2 * nd);
        }
        else
        {
            int k = 0, nin = 0;
            for (; k + 8 <= nd; k += 8)
            {
                const float4 a = dl4[k >> 2], c = dl4[(k >> 2) + 1];
                const float rr[8] = {md - a.x, md - a.y, md - a.z, md - a.w, md - c.x, md - c.y, md - c.z, md - c.w};
                unsigned in = 0;
#pragma unroll
                for (int j = 0; j < 8; j++) in |= ((rr[j] < d.huber_hi && rr[j] > -d.huber_hi) ? 1u : 0u) << j;
                nin += __popc(in);
#pragma unroll
                for (int j = 0; j < 8; j++)
                    sa = ((in >> j) & 1u) ? fmaf(2.0f, rr[j], sa) : (float)((double)sa + (rr[j] > 0 ? hp : hm));
            }
            for (; k < nd; k++)
            {
                const float rr = md - dl[k];
                const bool in = rr < d.huber_hi && rr > -d.huber_hi;
                nin += in ? 1 : 0;
                sa = in ? fmaf(2.0f, rr, sa) : (float)((double)sa + (rr > 0 ? hp : hm));
            }
            sb = (float)(2 * nin); // nin exact additions of 2
        }
        const float delta = (float)((double)(-sa) / ((double)sb + 10.0));
        md = md + delta;
        if (delta < F_0p01_HI && delta > -F_0p01_HI) break; // |delta| < 0.01 in double (:552)
    }
    d.seed[so + s] = make_float4(mn.x, mn.y, mn.z, md);
    d.seed_hl[so + s] = split_inverse(md);
    d.inv_md[so + s] = 1.0 / (double)md;
    d.tstable[so + s] = mn.w != 0.f ? DSM_STABLE : -1;
}

// -------------------------------------------------------------------------------------------
// K3+K4a  plane_gather — calculate_spaces_kernel (:644-662), calculate_pixels_norms_kernel (:664-712) and the
// window scan of calculate_sp_depth_norms_kernel (:792-863) fused on the same TMA-staged seed tile.
//
// The reference computes a normal for EVERY pixel and then reads the ones of a superpixel's inliers.  Here the
// window scan (half-warp per seed, lane = window row, membership / valid-depth / inlier masks) first compacts the
// INLIER pixel positions of each seed into shared memory; a second, dense phase (8 lanes per seed, 4 seeds per warp,
// every lane walks every 8th inlier) computes exactly those pixels' normals from the depth tile -- each inlier
// belongs to one seed, so no normal is computed twice and none is ever written to HBM (the 12 B/px `nrm` planes of
// the round-1 schedule are gone).  The same phase forms the back-projected points, their mean, the centred points
// (get_huber_norm :111-126, written as 32-byte runs of the per-seed lists qlist[b][seed][plane][PL_STRIDE]) and
// everything the first Gauss-Newton pass needs from the points: H = sum 2 q q^T over all points, the same sums over
// the points whose first residual is outside the Huber range (ho) with their clamped gradient (jo) (:133-171), the
// smallest distance of any |residual| to the range boundary and max |q|^2.  With these k_gn_solve takes its first
// step -- and, as long as the accumulated parameter change provably cannot move any residual across the boundary,
// every further step -- without touching the points.
// Pixel normal, fast path: n / |n| and the view angle with MUFU reciprocal square roots (a few ulp); the only place
// where the exact value matters is the `|view| < 0.1` skip test (:706), so a pixel whose view angle is within
// 1e-4 of +-0.1 is re-evaluated with the reference's IEEE divisions / square roots.
// Not label-affecting: float sums are lane-partial + tree (order-free within 1e-4, SURVEY.md H2/H5).
// -------------------------------------------------------------------------------------------
#define PL_STRIDE 232 // floats per plane of a seed's centred-point list (>= 225, multiple of 8)
#define HREC 24       // doubles per seed: H (9), ho (10), jo (4), packed (margin, qmax2)
#define PG_SMEM_DEP 0
#define PG_SMEM_COD TILE_PLANE_BYTES
#define PG_SMEM_POS (TILE_PLANE_BYTES + TILE_BYTE_PLANE)         // u16 [32][PG_POS_STRIDE]
#define PG_POS_STRIDE 232
#define PG_SMEM_KX (PG_SMEM_POS + 32 * PG_POS_STRIDE * 2)        // float [80] kx, float [48] ky
#define PG_SMEM_REC (PG_SMEM_KX + 128 * 4)                       // float maxd[32], int nvalid[32], int ninl[32]
#define PG_SMEM_BAR (PG_SMEM_REC + 96 * 4)
#define PG_SMEM_BYTES (PG_SMEM_BAR + 16)
#define PG_TX_BYTES (DSM_TILE_W * DSM_TILE_H * 4u + (unsigned)DSM_TILE_GW * DSM_TILE_H)

__device__ __forceinline__ float group8_sum_f(float v)
{
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ double group8_sum_d(double v)
{
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

__global__ void __launch_bounds__(256, 4) k_plane_gather(const __grid_constant__ DsmDev d, const __grid_constant__ DsmMaps mp)
{
    pdl_enter();
    extern __shared__ __align__(128) unsigned char smem[];
    const float *t_dep = reinterpret_cast<const float *>(smem + PG_SMEM_DEP);
    const uint8_t *t_cod = smem + PG_SMEM_COD;
    uint16_t *s_pos = reinterpret_cast<uint16_t *>(smem + PG_SMEM_POS);
    float *s_kx = reinterpret_cast<float *>(smem + PG_SMEM_KX), *s_ky = s_kx + 80;
    float *s_maxd = reinterpret_cast<float *>(smem + PG_SMEM_REC);
    int *s_nvalid = reinterpret_cast<int *>(s_maxd + 32), *s_ninl = s_nvalid + 32;
    const unsigned bar = smem_u32(smem + PG_SMEM_BAR);

    const int b = d.frame0 + blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int X0 = blockIdx.x * (DSM_TILE_SX * DSM_SP) - DSM_SP / 2, Y0 = blockIdx.y * (DSM_TILE_SY * DSM_SP) - DSM_SP / 2;
    if (threadIdx.x == 0)
    {
        mbar_init(bar, 1);
        mbar_expect_tx(bar, PG_TX_BYTES);
        tma_load_3d(smem_u32(smem + PG_SMEM_DEP), &mp.dep, X0, Y0, b, bar);
        tma_load_3d(smem_u32(smem + PG_SMEM_COD), &mp.cod, X0 - DSM_TILE_GX, Y0, b, bar);
    }
    const int W = d.W, H = d.H;
    const size_t so = (size_t)b * d.S;
    // back-projection factors of the tile's columns / rows (tables hold Wp+16 / H+16 entries; clamp the halo)
    if (threadIdx.x < 80)
    {
        int x = X0 + (int)threadIdx.x;
        x = x < 0 ? 0 : (x > d.Wp + 15 ? d.Wp + 15 : x);
        s_kx[threadIdx.x] = d.kx[x];
    }
    else if (threadIdx.x < 128)
    {
        int y = Y0 + (int)threadIdx.x - 80;
        y = y < 0 ? 0 : (y > H + 15 ? H + 15 : y);
        s_ky[threadIdx.x - 80] = d.ky[y];
    }
    const int half = lane >> 4, r = lane & 15;
    float4 sdv[2];
#pragma unroll
    for (int rd = 0; rd < 2; rd++)
    {
        const int sl = rd * 16 + warp * 2 + half;
        const int sp_x = blockIdx.x * DSM_TILE_SX + (sl & 7), sp_y = blockIdx.y * DSM_TILE_SY + (sl >> 3);
        const bool live = sp_x < d.spw && sp_y < d.sph;
        sdv[rd] = d.seed[so + (live ? sp_y * d.spw + sp_x : 0)]; // x, y, I, mean_depth (Huber mean after the 3 iterations)
    }
    __syncthreads();
    mbar_wait(bar, 0);
    // ---- phase 1: window scan, inlier positions in raster order
#pragma unroll
    for (int rd = 0; rd < 2; rd++)
    {
        const int sl = rd * 16 + warp * 2 + half;
        const int tx = sl & 7, ty = sl >> 3;
        const int sp_x = blockIdx.x * DSM_TILE_SX + tx, sp_y = blockIdx.y * DSM_TILE_SY + ty;
        const bool live = sp_x < d.spw && sp_y < d.sph;
        const float4 sd = sdv[rd];
        const int x0 = sp_x * DSM_SP - DSM_SP / 2, y0 = sp_y * DSM_SP - DSM_SP / 2;
        const int y = y0 + r;
        const bool rowin = live && y >= 0 && y < H; // window bounded by the flat index only (:816)
        const int kb = x0 < 0 ? -x0 : 0, ke = (W - x0) < 16 ? (W - x0) : 16;
        const unsigned kmask = rowin ? (((1u << ke) - 1u) & ~((1u << kb) - 1u)) : 0u;
        const int trow = ty * DSM_SP + r, tcol = tx * DSM_SP;
        unsigned mm, vm = 0, im = 0; // bit k: labelled with this seed / depth > 0.05 / |mean_depth - depth| < HUBER_RANGE
        {
            const unsigned *pc = reinterpret_cast<const unsigned *>(t_cod + trow * DSM_TILE_GW + DSM_TILE_GX + tcol); // 4-byte aligned
            const unsigned cw[4] = {pc[0], pc[1], pc[2], pc[3]};
            mm = member_mask16(cw, r);
            const float4 *pz = reinterpret_cast<const float4 *>(t_dep + trow * DSM_TILE_W + tcol);
#pragma unroll
            for (int qd = 0; qd < 4; qd++)
            {
                const float4 z = pz[qd];
                const float zz[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
                for (int j = 0; j < 4; j++)
                {
                    vm |= (zz[j] > F_0p05_LO ? 1u : 0u) << (4 * qd + j); // (double)depth > 0.05 (:827)
                    const float rr = sd.w - zz[j];
                    im |= ((rr < d.huber_hi && rr > -d.huber_hi) ? 1u : 0u) << (4 * qd + j); // inlier (:849-860)
                }
            }
        }
        mm &= kmask;
        vm &= mm;
        im &= vm;
        // max squared pixel distance of a member to the seed (:821-823): dist = fl(fl(xd^2) + fl(yd^2)) is monotone in |xd|,
        // so within the row it is attained at the leftmost or the rightmost member
        float maxd = 0.f;
        if (mm)
        {
            const float yd = (float)y - sd.y;
            const float yd2 = yd * yd;
            const float xl = (float)(x0 + __ffs(mm) - 1) - sd.x, xr = (float)(x0 + 31 - __clz(mm)) - sd.x;
            maxd = fmaxf(xl * xl + yd2, xr * xr + yd2);
        }
        int nvalid = __popc(vm);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1)
        {
            maxd = fmaxf(maxd, __shfl_xor_sync(FULL, maxd, o));
            nvalid += __shfl_xor_sync(FULL, nvalid, o);
        }
        const int c = __popc(im);
        int incl = c;
#pragma unroll
        for (int o = 1; o < 16; o <<= 1)
        {
            const int nb = __shfl_up_sync(FULL, incl, o, 16);
            if (r >= o) incl += nb;
        }
        const int ninl = __shfl_sync(FULL, incl, 15, 16);
        uint16_t *pp = s_pos + sl * PG_POS_STRIDE + (incl - c);
        const int pbase = (trow << 7) | tcol; // (tile row, tile column) packed: no division when unpacking
#pragma unroll
        for (int k = 0; k < 16; k++)
            if ((im >> k) & 1u) *pp++ = (uint16_t)(pbase + k);
        if (r == 0)
        {
            s_maxd[sl] = maxd;
            s_nvalid[sl] = nvalid;
            s_ninl[sl] = ninl;
        }
    }
    __syncthreads();
    // ---- phase 2: 8 lanes per seed, 4 seeds per warp; lane gl of a group walks the inliers gl, gl + 8, ...
    const int gl = lane & 7;
    const int sl = warp * 4 + (lane >> 3);
    const int sp_x = blockIdx.x * DSM_TILE_SX + (sl & 7), sp_y = blockIdx.y * DSM_TILE_SY + (sl >> 3);
    const bool live = sp_x < d.spw && sp_y < d.sph;
    const int s = sp_y * d.spw + sp_x;
    const int nvalid = s_nvalid[sl], ninl_raw = s_ninl[sl];
    const float maxd = s_maxd[sl];
    const bool ok = live && nvalid >= 16 && !((float)ninl_raw / (float)nvalid < F_0p8_HI); // (:841), (double)ratio < 0.8 (:862)
    const int ninl = ok ? ninl_raw : 0; // rejected seeds walk an empty list (the group stays convergent for the shuffles)
    const uint16_t *pos = s_pos + sl * PG_POS_STRIDE;
    float snx = 0.f, sny = 0.f, snz = 0.f, spx = 0.f, spy = 0.f, spz = 0.f;
    for (int j = gl; j < ninl; j += 8)
    {
        const int p = pos[j];
        const int trow = p >> 7, tcol = p & 127;
        const int x = X0 + tcol, y = Y0 + trow;
        const float *pz = t_dep + trow * DSM_TILE_W + tcol;
        const float mz = pz[0];
        const float kxi = s_kx[tcol], ky0 = s_ky[trow];
        const float mx = kxi * mz, my = ky0 * mz; // back_project in float (:94-96)
        spx += mx;
        spy += my;
        spz += mz;
        // pixel normal of (x, y), as calculate_pixels_norms_kernel (:664-712)
        if (y >= 1 && y <= H - 2 && x >= 1 && x <= W - 2)
        {
            const float rz = pz[1], dz = pz[DSM_TILE_W];
            if (!(mz < F_0p1_HI || rz < F_0p1_HI || dz < F_0p1_HI)) // (double)z < 0.1 (:688)
            {
                const float kxr = s_kx[tcol + 1], ky1 = s_ky[trow + 1];
                const float rx = kxr * rz - mx, ry = ky0 * rz - my, rzz = rz - mz;
                const float dx = kxi * dz - mx, dy = ky1 * dz - my, dzz = dz - mz;
                float cxn = ry * dzz - rzz * dy;
                float cyn = rzz * dx - rx * dzz;
                float czn = rx * dy - ry * dx;
                const float l2 = cxn * cxn + cyn * cyn + czn * czn, p2 = mx * mx + my * my + mz * mz;
                const float il = rsqrtf(l2);
                float nx = cxn * il, ny = cyn * il, nz = czn * il;
                float view = (nx * mx + ny * my + nz * mz) * rsqrtf(p2);
                const float av = fabsf(view);
                if (!(av > 0.1001f || av < 0.0999f))
                { // within 1e-4 of the skip threshold (or NaN): the reference's own arithmetic decides
                    const float len = sqrtf(l2);
                    nx = cxn / len, ny = cyn / len, nz = czn / len;
                    view = (nx * mx + ny * my + nz * mz) / sqrtf(p2);
                }
                if (!(view > -F_0p1_HI && view < F_0p1_HI)) // |view| < 0.1 in double -> skipped (:706)
                    snx += nx, sny += ny, snz += nz;
            }
        }
    }
    snx = group8_sum_f(snx), sny = group8_sum_f(sny), snz = group8_sum_f(snz);
    spx = group8_sum_f(spx), spy = group8_sum_f(spy), spz = group8_sum_f(spz);
    const float fn = (float)ninl;
    const float mxs = spx / fn, mys = spy / fn, mzs = spz / fn; // (:117-119)
    // initial normal of get_huber_norm = normalised sum of the inlier pixel normals (:864-871); 0/0 -> NaN, propagated (H6-iii)
    const float len0 = sqrtf(snx * snx + sny * sny + snz * snz);
    const float n0x = snx / len0, n0y = sny / len0, n0z = snz / len0;
    double h[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}; // xx xy xz xw yy yz yw zz zw over all points
    float margin = __int_as_float(0x7f800000), qmax2 = 0.f;
    bool rnan = false;
    unsigned omask = 0; // bit i: this lane's i-th point (j = gl + 8 i, i <= 28) is outside the Huber range
    float *qx = d.qlist + (so + s) * (3 * PL_STRIDE), *qy = qx + PL_STRIDE, *qz = qy + PL_STRIDE;
    for (int j = gl, it = 0; j < ninl; j += 8, it++)
    {
        const int p = pos[j];
        const int trow = p >> 7, tcol = p & 127;
        const float mz = t_dep[trow * DSM_TILE_W + tcol];
        const float ax = s_kx[tcol] * mz - mxs, ay = s_ky[trow] * mz - mys, az = mz - mzs; // centred points (:121-126)
        qx[j] = ax, qy[j] = ay, qz[j] = az;
        const float rr = ax * n0x + ay * n0y + az * n0z + 0.f; // first-pass residual (:133), b = 0
        rnan |= !(rr == rr);
        margin = fminf(margin, fabsf(fabsf(rr) - d.huber_hi));
        qmax2 = fmaxf(qmax2, ax * ax + ay * ay + az * az);
        h[0] += (double)(2 * ax * ax), h[1] += (double)(2 * ax * ay), h[2] += (double)(2 * ax * az), h[3] += (double)(2 * ax);
        h[4] += (double)(2 * ay * ay), h[5] += (double)(2 * ay * az), h[6] += (double)(2 * ay);
        h[7] += (double)(2 * az * az), h[8] += (double)(2 * az);
        if (!(rr < d.huber_hi && rr > -d.huber_hi)) omask |= 1u << it; // (:134)
    }
#pragma unroll
    for (int i = 0; i < 9; i++) h[i] = group8_sum_d(h[i]);
#pragma unroll
    for (int o = 4; o > 0; o >>= 1)
    {
        margin = fminf(margin, __shfl_xor_sync(FULL, margin, o));
        qmax2 = fmaxf(qmax2, __shfl_xor_sync(FULL, qmax2, o));
        rnan |= __shfl_xor_sync(FULL, rnan ? 1 : 0, o) != 0;
    }
    if (rnan) margin = __int_as_float(0x7fc00000); // a NaN residual: no pass may ever be skipped
    double *hr = d.hrec + (size_t)b * HREC * d.S + s; // [b][field][seed]: the solver's thread-per-seed reads coalesce
    const size_t hs = (size_t)d.S;
    if (ok)
    { // the group's lanes write the 9 sums and the packed (margin, qmax2)
#pragma unroll
        for (int i = 0; i < 9; i++)
            if ((i & 7) == gl) hr[i * hs] = h[i];
        if (gl == 7) hr[23 * hs] = __hiloint2double(__float_as_int(qmax2), __float_as_int(margin));
    }
    // the out-of-range points (few per seed, none for most): the same ten sums (with ww) and the clamped gradient
    // (:157-170), accumulated in a second sweep over just those points so that the 14 accumulators are not live above
    double ho[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, jo[4] = {0, 0, 0, 0};
    if (__any_sync(FULL, omask != 0)) // warp-uniform
    {
        while (omask)
        {
            const int it = __ffs(omask) - 1;
            omask &= omask - 1;
            const int p = pos[gl + 8 * it];
            const int trow = p >> 7, tcol = p & 127;
            const float mz = t_dep[trow * DSM_TILE_W + tcol];
            const float ax = s_kx[tcol] * mz - mxs, ay = s_ky[trow] * mz - mys, az = mz - mzs;
            const float rr = ax * n0x + ay * n0y + az * n0z + 0.f;
            ho[0] += (double)(2 * ax * ax), ho[1] += (double)(2 * ax * ay), ho[2] += (double)(2 * ax * az), ho[3] += (double)(2 * ax);
            ho[4] += (double)(2 * ay * ay), ho[5] += (double)(2 * ay * az), ho[6] += (double)(2 * ay);
            ho[7] += (double)(2 * az * az), ho[8] += (double)(2 * az), ho[9] += 2;
            if (rr >= d.huber_hi)
            { // (double)r >= 0.4 (:157-163)
                jo[0] += d.huber * (double)ax, jo[1] += d.huber * (double)ay, jo[2] += d.huber * (double)az, jo[3] += d.huber;
            }
            else if (rr <= -d.huber_hi)
            { // (double)r <= -0.4 (:164-170)
                jo[0] += -1 * d.huber * (double)ax, jo[1] += -1 * d.huber * (double)ay, jo[2] += -1 * d.huber * (double)az,
                    jo[3] += -1 * d.huber;
            }
        }
#pragma unroll
        for (int i = 0; i < 10; i++) ho[i] = group8_sum_d(ho[i]);
#pragma unroll
        for (int i = 0; i < 4; i++) jo[i] = group8_sum_d(jo[i]);
    }
    if (ok)
    { // hr[18] = ho[9] (twice the number of out-of-range points) doubles as the "any" flag the solver tests
        if (ho[9] != 0.0)
        {
#pragma unroll
            for (int i = 0; i < 14; i++)
                if ((i & 7) == gl) hr[(9 + i) * hs] = i < 10 ? ho[i] : jo[i - 10];
        }
        else if (gl == 0)
            hr[18 * hs] = 0.0;
    }
    if (live && gl == 0)
    {
        d.pfsum[(so + s) * 2] = ok ? make_float4(snx, sny, snz, maxd) : make_float4(0.f, 0.f, 0.f, maxd);
        d.pfsum[(so + s) * 2 + 1] = ok ? make_float4(mxs, mys, mzs, __int_as_float(ninl)) : make_float4(0.f, 0.f, 0.f, __int_as_float(0));
    }
}

// -------------------------------------------------------------------------------------------
// K4b  plane_solve — get_huber_norm (:104-188) + the projection (:884-912), one thread per seed.
// Algebra: the reference rebuilds H = sum w q~ q~^T and J = sum w r q~ (q~ = (q, 1), theta = (n, b)) from the points in
// every pass (:131-171).  For the points whose residual is inside the Huber range,
// sum 2 r q~ = (sum 2 q~ q~^T) theta, so with H over ALL points, H_R = H - ho and J = H_R theta + jo, where ho / jo are
// the sums over the out-of-range points only.  A pass over the points is needed only to find out which points are
// out of range.  Let m = min_i | |r_i| - 0.4 | at the last evaluated parameters; a step (dn, db) changes every
// residual by at most |q|max |dn| + |db|, so while the accumulated bound stays below m (minus a slack far above the
// float error of evaluating r) no point crosses the boundary: ho, jo are provably unchanged and the pass is skipped.
// The first pass's sums arrive from k_plane_gather, so most seeds are five register-only 4x4 solves; the others read
// the centred points from qlist[b][seed][plane][k] (16-byte loads) exactly like the reference's loop (:131-171).
// -------------------------------------------------------------------------------------------
__device__ __forceinline__ void solve4_spd_t(const double *h, double lambda, const double *j, double *u)
{ // h: 10 unique entries xx xy xz xw yy yz yw zz zw ww of an SPD matrix; solves (H + lambda I) u = j
    const double a00 = h[0] + lambda, a01 = h[1], a02 = h[2], a03 = h[3];
    const double i0 = 1.0 / a00;
    const double l10 = a01 * i0, l20 = a02 * i0, l30 = a03 * i0;
    const double a11 = (h[4] + lambda) - l10 * a01, a12 = h[5] - l10 * a02, a13 = h[6] - l10 * a03;
    const double a22p = (h[7] + lambda) - l20 * a02, a23p = h[8] - l20 * a03, a33p = (h[9] + lambda) - l30 * a03;
    const double i1 = 1.0 / a11;
    const double l21 = a12 * i1, l31 = a13 * i1;
    const double a22 = a22p - l21 * a12, a23 = a23p - l21 * a13, a33q = a33p - l31 * a13;
    const double i2 = 1.0 / a22;
    const double l32 = a23 * i2;
    const double a33 = a33q - l32 * a23;
    const double y0 = j[0];
    const double y1 = j[1] - l10 * y0;
    const double y2 = j[2] - l20 * y0 - l21 * y1;
    const double y3 = j[3] - l30 * y0 - l31 * y1 - l32 * y2;
    u[3] = y3 / a33;
    u[2] = y2 * i2 - l32 * u[3];
    u[1] = y1 * i1 - l21 * u[2] - l31 * u[3];
    u[0] = y0 * i0 - l10 * u[1] - l20 * u[2] - l30 * u[3];
}

// centre of the superpixel projected onto the fitted plane, view angle, size (:872-912): the seed's final record
__device__ __forceinline__ void finish_plane(const DsmDev &d, size_t o, const float4 &sd, const float4 &P0, const float4 &P1, float nx, float ny,
                                             float nz, float nb)
{
    nb = nb - (nx * P1.x + ny * P1.y + nz * P1.z);
    const float nl = sqrtf(nx * nx + ny * ny + nz * nz);
    nx /= nl;
    ny /= nl;
    nz /= nl;
    nb /= nl;
    const float axf = (sd.x - d.cx) / d.fx * sd.w;
    const float ayf = (sd.y - d.cy) / d.fy * sd.w;
    double ax = (double)axf, ay = (double)ayf, az = (double)sd.w;
    const float kk = (float)(-1 * (ax * (double)nx + ay * (double)ny + az * (double)nz) - (double)nb);
    ax += (double)(kk * nx);
    ay += (double)(kk * ny);
    az += (double)(kk * nz);
    const float mean_depth = (float)az;
    float view_cos = (float)(-1.0 * ((double)nx * ax + (double)ny * ay + (double)nz * az) / sqrt(ax * ax + ay * ay + az * az));
    if (view_cos < 0)
    {
        view_cos = -view_cos;
        nx = -nx;
        ny = -ny;
        nz = -nz;
    }
    float4 *pl = d.plane + o * 3;
    pl[0] = make_float4(nx, ny, nz, view_cos);
    pl[1] = make_float4((float)ax, (float)ay, (float)az, mean_depth);
    pl[2] = make_float4(sqrtf(P0.w), sd.z, sd.x, sd.y);
}

// one damped Gauss-Newton step (:172-181) from hh0 = H over the in-range points and jo = clamped gradient of the others;
// returns the bound on how far the step can move any residual: |q|max |dn| + |db| (+ rounding slack)
__device__ __forceinline__ float gn_step(const double *hh0, const double *jo, float qmax, float &nx, float &ny, float &nz, float &nb)
{
    double jj[4];
    const double tx = (double)nx, ty = (double)ny, tz = (double)nz, tb = (double)nb;
    jj[0] = ((hh0[0] * tx + hh0[1] * ty) + hh0[2] * tz) + hh0[3] * tb + jo[0];
    jj[1] = ((hh0[1] * tx + hh0[4] * ty) + hh0[5] * tz) + hh0[6] * tb + jo[1];
    jj[2] = ((hh0[2] * tx + hh0[5] * ty) + hh0[7] * tz) + hh0[8] * tb + jo[2];
    jj[3] = ((hh0[3] * tx + hh0[6] * ty) + hh0[8] * tz) + hh0[9] * tb + jo[3];
    double u[4];
    solve4_spd_t(hh0, 5.0, jj, u); // LM damping: + 5 on the diagonal (:172-175)
    const float ox = nx, oy = ny, oz = nz, ob = nb;
    nx = (float)((double)nx - u[0]);
    ny = (float)((double)ny - u[1]);
    nz = (float)((double)nz - u[2]);
    nb = (float)((double)nb - u[3]);
    const float dx = nx - ox, dy = ny - oy, dz = nz - oz;
    return qmax * sqrtf(dx * dx + dy * dy + dz * dz) * 1.0001f + fabsf(nb - ob) + 1e-4f;
}

#define GS_CAP 9216 // floats of point staging per 128-seed CTA (36 KB): three planes of the queued seeds' centred points
__global__ void __launch_bounds__(128, 4) k_gn_solve(const __grid_constant__ DsmDev d)
{
    pdl_enter();
    // Phase A: every seed iterates from the sums of k_plane_gather for as long as no residual can have crossed the Huber
    // boundary -- most seeds finish all five steps here without ever touching their points.  A seed that has to classify
    // its points again is queued.  Phase B: the queued seeds' point lists (contiguous runs in global memory) are staged
    // into shared memory with cp.async and the seeds continue, packed densely into the CTA's first warps.
    __shared__ __align__(16) float pts[GS_CAP];
    __shared__ float4 s_theta[128]; // queued seed: plane parameters so far
    __shared__ int s_queue[128], s_gn[128], s_poff[128], s_nq, s_used;
    const int b = d.frame0 + blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = blockIdx.x * 128 + tid;
    const size_t so = (size_t)b * d.S;
    const size_t hs = (size_t)d.S;
    if (tid == 0) s_nq = 0, s_used = 0;
    __syncthreads();
    if (s < d.S)
    {
        const float4 sd = d.seed[so + s];
        const float4 P0 = d.pfsum[(so + s) * 2], P1 = d.pfsum[(so + s) * 2 + 1];
        const int n = __float_as_int(P1.w);
        if (n <= 0)
        { // plane fit rejected -> zero normal / position / view_cos / size (H6-i), Huber mean depth kept
            float4 *pl = d.plane + (so + s) * 3;
            pl[0] = make_float4(0.f, 0.f, 0.f, 0.f);
            pl[1] = make_float4(0.f, 0.f, 0.f, sd.w);
            pl[2] = make_float4(0.f, sd.z, sd.x, sd.y);
        }
        else
        {
            const float len0 = sqrtf(P0.x * P0.x + P0.y * P0.y + P0.z * P0.z);
            float nx = P0.x / len0, ny = P0.y / len0, nz = P0.z / len0, nb = 0.f; // len0 == 0 -> NaN, propagated (H6-iii)
            const double *hr = d.hrec + (size_t)b * HREC * d.S + s; // [b][field][seed]
            // hh0 = H over the in-range points = H_all - ho; jo = clamped gradient of the out-of-range points
            double hh0[10], jo[4] = {0, 0, 0, 0};
#pragma unroll
            for (int i = 0; i < 9; i++) hh0[i] = hr[i * hs];
            hh0[9] = 2.0 * (double)n;
            if (hr[18 * hs] != 0.0)
            { // the first pass found points outside the Huber range
#pragma unroll
                for (int i = 0; i < 10; i++) hh0[i] -= hr[(9 + i) * hs];
#pragma unroll
                for (int i = 0; i < 4; i++) jo[i] = hr[(19 + i) * hs];
            }
            const double pk = hr[23 * hs];
            const float margin = __int_as_float(__double2loint(pk));
            const float qmax = sqrtf(__int_as_float(__double2hiint(pk)));
            float moved = 0.f; // bound on the change of any residual since the classification behind hh0 / jo was made
            int gn = 0;
            for (; gn < 5; gn++)
            {
                if (gn > 0 && !(moved + 2e-3f < margin)) break; // NaN-safe: a NaN margin queues the seed
                moved += gn_step(hh0, jo, qmax, nx, ny, nz, nb);
            }
            if (gn == 5)
                finish_plane(d, so + s, sd, P0, P1, nx, ny, nz, nb);
            else
            { // some point may have crossed the Huber boundary: continue in phase B
                const int q = atomicAdd(&s_nq, 1);
                const int len4 = (n + 3) & ~3;
                const int off = atomicAdd(&s_used, 3 * len4);
                s_queue[q] = tid;
                s_gn[tid] = gn;
                s_poff[tid] = (off + 3 * len4 <= GS_CAP) ? off : -1;
                s_theta[tid] = make_float4(nx, ny, nz, nb);
            }
        }
    }
    __syncthreads();
    const int nq = s_nq;
    if (nq == 0) return;
    for (int q = warp; q < nq; q += 4)
    { // stage the three planes of a queued seed's centred points: coalesced 16-byte cp.async, all in flight at once
        const int t2 = s_queue[q], off = s_poff[t2];
        if (off < 0) continue; // does not fit: that seed reads global memory
        const size_t o2 = so + blockIdx.x * 128 + t2;
        const int n2 = __float_as_int(d.pfsum[o2 * 2 + 1].w), l4 = ((n2 + 3) & ~3) >> 2;
        const float4 *src = reinterpret_cast<const float4 *>(d.qlist + o2 * (3 * PL_STRIDE));
        float4 *dst = reinterpret_cast<float4 *>(pts + off);
        for (int pln = 0; pln < 3; pln++)
            for (int j4 = lane; j4 < l4; j4 += 32) __pipeline_memcpy_async(dst + pln * l4 + j4, src + pln * (PL_STRIDE / 4) + j4, 16);
    }
    __pipeline_commit();
    __pipeline_wait_prior(0);
    __syncthreads();
    for (int q = tid; q < nq; q += 128)
    {
        const int t2 = s_queue[q];
        const size_t o2 = so + blockIdx.x * 128 + t2;
        const float4 sd = d.seed[o2];
        const float4 P0 = d.pfsum[o2 * 2], P1 = d.pfsum[o2 * 2 + 1];
        const int n = __float_as_int(P1.w), l4 = ((n + 3) & ~3) >> 2;
        const double *hr = d.hrec + (size_t)b * HREC * d.S + (blockIdx.x * 128 + t2);
        const float qmax = sqrtf(__int_as_float(__double2hiint(hr[23 * hs])));
        const float4 th = s_theta[t2];
        float nx = th.x, ny = th.y, nz = th.z, nb = th.w;
        const int off = s_poff[t2];
        const float4 *qx = off >= 0 ? reinterpret_cast<const float4 *>(pts + off) : reinterpret_cast<const float4 *>(d.qlist + o2 * (3 * PL_STRIDE));
        const int pstride = off >= 0 ? l4 : PL_STRIDE / 4; // float4 units between the planes
        float margin = 0.f, moved = 0.f;
        double hh0[10], jo[4];
        for (int gn = s_gn[t2]; gn < 5; gn++)
        {
            if (!(moved + 2e-3f < margin))
            { // classify the points again (:131-171)
#pragma unroll
                for (int i = 0; i < 9; i++) hh0[i] = hr[i * hs];
                hh0[9] = 2.0 * (double)n;
#pragma unroll
                for (int i = 0; i < 4; i++) jo[i] = 0.0;
                float mg = __int_as_float(0x7f800000);
                bool rnan = false;
                auto point = [&](float ax, float ay, float az)
                {
                    const float r = ax * nx + ay * ny + az * nz + nb; // (:133)
                    rnan |= !(r == r);
                    mg = fminf(mg, fabsf(fabsf(r) - d.huber_hi));
                    if (!(r < d.huber_hi && r > -d.huber_hi)) // (:134)
                    {
                        hh0[0] -= (double)(2 * ax * ax), hh0[1] -= (double)(2 * ax * ay), hh0[2] -= (double)(2 * ax * az), hh0[3] -= (double)(2 * ax);
                        hh0[4] -= (double)(2 * ay * ay), hh0[5] -= (double)(2 * ay * az), hh0[6] -= (double)(2 * ay);
                        hh0[7] -= (double)(2 * az * az), hh0[8] -= (double)(2 * az), hh0[9] -= 2;
                        if (r >= d.huber_hi)
                        { // (double)r >= HUBER_RANGE (:157-163)
                            jo[0] += d.huber * (double)ax, jo[1] += d.huber * (double)ay;
                            jo[2] += d.huber * (double)az, jo[3] += d.huber;
                        }
                        else if (r <= -d.huber_hi)
                        { // (double)r <= -HUBER_RANGE (:164-170)
                            jo[0] += -1 * d.huber * (double)ax, jo[1] += -1 * d.huber * (double)ay;
                            jo[2] += -1 * d.huber * (double)az, jo[3] += -1 * d.huber;
                        }
                    }
                };
                int k = 0;
                for (; k + 4 <= n; k += 4)
                {
                    const float4 a = qx[k >> 2], bb = qx[pstride + (k >> 2)], c = qx[2 * pstride + (k >> 2)];
                    point(a.x, bb.x, c.x);
                    point(a.y, bb.y, c.y);
                    point(a.z, bb.z, c.z);
                    point(a.w, bb.w, c.w);
                }
                if (k < n)
                {
                    const float4 a = qx[k >> 2], bb = qx[pstride + (k >> 2)], c = qx[2 * pstride + (k >> 2)];
                    point(a.x, bb.x, c.x);
                    if (k + 1 < n) point(a.y, bb.y, c.y);
                    if (k + 2 < n) point(a.z, bb.z, c.z);
                }
                margin = rnan ? __int_as_float(0x7fc00000) : mg;
                moved = 0.f;
            }
            moved += gn_step(hh0, jo, qmax, nx, ny, nz, nb);
        }
        finish_plane(d, o2, sd, P0, P1, nx, ny, nz, nb);
    }
}

// -------------------------------------------------------------------------------------------
// launchers
// -------------------------------------------------------------------------------------------
int dsm_tile_setup()
{
    cudaError_t e = cudaFuncSetAttribute(k_gather, cudaFuncAttributeMaxDynamicSharedMemorySize, GAT_SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_plane_gather, cudaFuncAttributeMaxDynamicSharedMemorySize, PG_SMEM_BYTES);
    // shared memory is what limits the residency of the two tile kernels (36.6 KB / 33 KB per CTA): ask for the largest carve-out;
    // k_gather then runs 6 CTAs per SM (measured 60.5 -> 55.5 us per launch; 5 CTAs for k_plane_gather gave nothing)
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_gather, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_plane_gather, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    return e == cudaSuccess ? 0 : -1;
}
void dsm_launch_assign2(const DsmDev &d, int nb, bool first, cudaStream_t s)
{
    // one CTA per seed-row band (pixel rows 8k-4 .. 8k+3) and 128-column run (starting at 128a - 4)
    dim3 block(ASG_TX, 8);
    dim3 grid((d.W + 4 + 8 * ASG_TX - 1) / (8 * ASG_TX), (d.H + 4 + 7) / 8, nb);
    if (first)
        pdl_launch(k_assign2<true>, grid, block, 0, s, d);
    else
        pdl_launch(k_assign2<false>, grid, block, 0, s, d);
}
void dsm_launch_gather(const DsmDev &d, const DsmMaps &m, int nb, cudaStream_t s)
{
    dim3 grid((d.spw + DSM_TILE_SX - 1) / DSM_TILE_SX, (d.sph + DSM_TILE_SY - 1) / DSM_TILE_SY, nb);
    pdl_launch(k_gather, grid, dim3(256), GAT_SMEM_BYTES, s, d, m);
}
void dsm_launch_newton2(const DsmDev &d, int nb, cudaStream_t s)
{
    dim3 grid((d.S + NW_T - 1) / NW_T, nb);
    pdl_launch(k_newton2, grid, dim3(NW_T), 0, s, d);
    pdl_launch(k_newton_hard, grid, dim3(NW_T), 0, s, d); // surplus CTAs exit at once: the queue length is on the device
}
void dsm_launch_plane_gather(const DsmDev &d, const DsmMaps &m, int nb, cudaStream_t s)
{
    dim3 grid((d.spw + DSM_TILE_SX - 1) / DSM_TILE_SX, (d.sph + DSM_TILE_SY - 1) / DSM_TILE_SY, nb);
    pdl_launch(k_plane_gather, grid, dim3(256), PG_SMEM_BYTES, s, d, m);
}
void dsm_launch_gn_solve(const DsmDev &d, int nb, cudaStream_t s)
{
    dim3 grid((d.S + 127) / 128, nb);
    pdl_launch(k_gn_solve, grid, dim3(128), 0, s, d);
}
