// vap_format.cuh -- "next" row f1: text of the trajectory export on the device.
//
// The reference writes every value with f"{v} " (gui_manager.py:220-230), i.e. Python's repr(float): the SHORTEST decimal
// string that round-trips, closest to the true value, laid out by float_repr_style 'short' (fixed notation for
// 1e-4 <= |x| < 1e16, otherwise d.ddde+XX).  Shortest digits are produced with the Ryu construction (Adams, PLDI 2018):
// one 64 x 128-bit multiplication by a tabulated 125-bit power of five gives the scaled value and its two neighbours'
// midpoints, digits are stripped while the interval still contains a shorter number.  Tables: vap_pow5_tables.cuh.
// Pinned against CPython's own formatting on random bit patterns and on the golden trajectories (tests/test_next_rows.py).
#pragma once
#include <cstdint>
#include "vap_pow5_tables.cuh"

__device__ __forceinline__ uint32_t f_pow5bits(int32_t e) { return (uint32_t)(((e * 1217359) >> 19) + 1); }     // bitlen(5^e)
__device__ __forceinline__ uint32_t f_log10pow2(int32_t e) { return ((uint32_t)e * 78913u) >> 18; }              // floor(e log10 2)
__device__ __forceinline__ uint32_t f_log10pow5(int32_t e) { return ((uint32_t)e * 732923u) >> 20; }             // floor(e log10 5)

__device__ __forceinline__ uint64_t f_mulshift(uint64_t m, const uint64_t* mul, int32_t j)
{   // (m * mul) >> j for 64 <= j < 128 + 64, mul = mul[0] + 2^64 mul[1]
    unsigned __int128 b0 = (unsigned __int128)m * __ldg(mul);
    unsigned __int128 b2 = (unsigned __int128)m * __ldg(mul + 1);
    return (uint64_t)(((b0 >> 64) + b2) >> (j - 64));
}
__device__ __forceinline__ bool f_mult_pow5(uint64_t v, uint32_t p)
{
    uint32_t c = 0;
    while (v != 0 && v % 5 == 0) { v /= 5; c++; if (c >= p) return true; }
    return c >= p;
}
__device__ __forceinline__ bool f_mult_pow2(uint64_t v, uint32_t p) { return (v & ((1ull << p) - 1)) == 0; }

// shortest decimal of a finite, non-zero double given by its fields: value = digits * 10^exp10
__device__ void shortest_decimal(uint64_t ieee_m, uint32_t ieee_e, uint64_t& digits, int32_t& exp10)
{
    int32_t e2;
    uint64_t m2;
    if (ieee_e == 0) { e2 = 1 - 1023 - 52 - 2; m2 = ieee_m; }
    else { e2 = (int32_t)ieee_e - 1023 - 52 - 2; m2 = (1ull << 52) | ieee_m; }
    const bool accept = (m2 & 1) == 0;
    const uint64_t mv = 4 * m2;
    const uint32_t mm_shift = (ieee_m != 0 || ieee_e <= 1) ? 1u : 0u;
    uint64_t vr, vp, vm;
    int32_t e10;
    bool vm_tz = false, vr_tz = false;
    if (e2 >= 0) {
        const uint32_t q = f_log10pow2(e2) - (e2 > 3);
        e10 = (int32_t)q;
        const int32_t k = VAP_POW5_BITS + (int32_t)f_pow5bits((int32_t)q) - 1;
        const int32_t i = -e2 + (int32_t)q + k;
        const uint64_t* mul = &VAP_POW5_INV[q][0];
        vr = f_mulshift(4 * m2, mul, i);
        vp = f_mulshift(4 * m2 + 2, mul, i);
        vm = f_mulshift(4 * m2 - 1 - mm_shift, mul, i);
        if (q <= 21) {
            if (mv % 5 == 0) vr_tz = f_mult_pow5(mv, q);
            else if (accept) vm_tz = f_mult_pow5(mv - 1 - mm_shift, q);
            else vp -= f_mult_pow5(mv + 2, q);
        }
    } else {
        const uint32_t q = f_log10pow5(-e2) - (-e2 > 1);
        e10 = (int32_t)q + e2;
        const int32_t i = -e2 - (int32_t)q;
        const int32_t k = (int32_t)f_pow5bits(i) - VAP_POW5_BITS;
        const int32_t j = (int32_t)q - k;
        const uint64_t* mul = &VAP_POW5[i][0];
        vr = f_mulshift(4 * m2, mul, j);
        vp = f_mulshift(4 * m2 + 2, mul, j);
        vm = f_mulshift(4 * m2 - 1 - mm_shift, mul, j);
        if (q <= 1) {
            vr_tz = true;
            if (accept) vm_tz = mm_shift == 1;
            else --vp;
        } else if (q < 63) {
            vr_tz = f_mult_pow2(mv, q);
        }
    }
    int32_t removed = 0;
    uint32_t last = 0;
    uint64_t out;
    if (vm_tz || vr_tz) {
        for (;;) {
            const uint64_t vp10 = vp / 10, vm10 = vm / 10;
            if (vp10 <= vm10) break;
            const uint32_t vmm = (uint32_t)(vm - 10 * vm10);
            const uint64_t vr10 = vr / 10;
            const uint32_t vrm = (uint32_t)(vr - 10 * vr10);
            vm_tz &= vmm == 0;
            vr_tz &= last == 0;
            last = vrm;
            vr = vr10; vp = vp10; vm = vm10; ++removed;
        }
        if (vm_tz) {
            for (;;) {
                const uint64_t vm10 = vm / 10;
                const uint32_t vmm = (uint32_t)(vm - 10 * vm10);
                if (vmm != 0) break;
                const uint64_t vp10 = vp / 10, vr10 = vr / 10;
                const uint32_t vrm = (uint32_t)(vr - 10 * vr10);
                vr_tz &= last == 0;
                last = vrm;
                vr = vr10; vp = vp10; vm = vm10; ++removed;
            }
        }
        if (vr_tz && last == 5 && vr % 2 == 0) last = 4;          // exactly half: round to even
        out = vr + (((vr == vm && (!accept || !vm_tz)) || last >= 5) ? 1 : 0);
    } else {
        bool up = false;
        const uint64_t vp100 = vp / 100, vm100 = vm / 100;
        if (vp100 > vm100) {
            const uint64_t vr100 = vr / 100;
            up = (uint32_t)(vr - 100 * vr100) >= 50;
            vr = vr100; vp = vp100; vm = vm100; removed += 2;
        }
        for (;;) {
            const uint64_t vp10 = vp / 10, vm10 = vm / 10;
            if (vp10 <= vm10) break;
            const uint64_t vr10 = vr / 10;
            up = (uint32_t)(vr - 10 * vr10) >= 5;
            vr = vr10; vp = vp10; vm = vm10; ++removed;
        }
        out = vr + ((vr == vm || up) ? 1 : 0);
    }
    digits = out;
    exp10 = e10 + removed;
}

// repr(float) into buf (at most 24 characters); returns the length
__device__ int format_repr(double x, char* buf)
{
    const uint64_t bits = (uint64_t)__double_as_longlong(x);
    const bool neg = (bits >> 63) != 0;
    const uint64_t m = bits & ((1ull << 52) - 1);
    const uint32_t e = (uint32_t)((bits >> 52) & 0x7ff);
    int n = 0;
    if (e == 0x7ff) {
        if (m != 0) { buf[0] = 'n'; buf[1] = 'a'; buf[2] = 'n'; return 3; }
        if (neg) buf[n++] = '-';
        buf[n++] = 'i'; buf[n++] = 'n'; buf[n++] = 'f';
        return n;
    }
    if (neg) buf[n++] = '-';
    if (e == 0 && m == 0) { buf[n++] = '0'; buf[n++] = '.'; buf[n++] = '0'; return n; }
    uint64_t dig;
    int32_t ex;
    shortest_decimal(m, e, dig, ex);
    char d[20];
    int nd = 0;
    while (dig != 0) { d[nd++] = (char)('0' + (int)(dig % 10)); dig /= 10; }     // reversed
    const int decpt = nd + ex;                                                    // value = 0.DIGITS * 10^decpt
    if (decpt > 16 || decpt <= -4) {                                              // float_repr_style 'short', repr
        buf[n++] = d[nd - 1];
        if (nd > 1) { buf[n++] = '.'; for (int i = nd - 2; i >= 0; i--) buf[n++] = d[i]; }
        buf[n++] = 'e';
        int xe = decpt - 1;
        if (xe < 0) { buf[n++] = '-'; xe = -xe; } else buf[n++] = '+';
        if (xe >= 100) { buf[n++] = (char)('0' + xe / 100); xe %= 100; buf[n++] = (char)('0' + xe / 10); buf[n++] = (char)('0' + xe % 10); }
        else { buf[n++] = (char)('0' + xe / 10); buf[n++] = (char)('0' + xe % 10); }
        return n;
    }
    if (decpt <= 0) {
        buf[n++] = '0'; buf[n++] = '.';
        for (int i = 0; i < -decpt; i++) buf[n++] = '0';
        for (int i = nd - 1; i >= 0; i--) buf[n++] = d[i];
    } else if (decpt >= nd) {
        for (int i = nd - 1; i >= 0; i--) buf[n++] = d[i];
        for (int i = 0; i < decpt - nd; i++) buf[n++] = '0';
        buf[n++] = '.'; buf[n++] = '0';
    } else {
        for (int i = nd - 1; i >= nd - decpt; i--) buf[n++] = d[i];
        buf[n++] = '.';
        for (int i = nd - decpt - 1; i >= 0; i--) buf[n++] = d[i];
    }
    return n;
}

#ifndef VAP_FORMAT_HOST_TEST
// n doubles -> fixed 32-byte slots (repr text, NUL padded) + lengths
__global__ void __launch_bounds__(256) k_format_doubles(long long n, const double* __restrict__ x, char* __restrict__ out,
                                                        int* __restrict__ lens)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    char buf[32];
    int len = format_repr(x[i], buf);
    for (int k = len; k < 32; k++) buf[k] = 0;
    uint4* o = reinterpret_cast<uint4*>(out + (size_t)i * 32);
    const uint4* s = reinterpret_cast<const uint4*>(buf);
    o[0] = s[0]; o[1] = s[1];
    lens[i] = len;
}

// Export rows -> text.  rows[R][7] = {0, t, x*12, y*-12, heading, v*12, omega}; every value is followed by one blank, the
// row ends with '\n' (fill_txt_file).  Column 0 is the integer 0.  kinds[r] (the RK_* bits of k_row_kinds) says which other
// columns hold a Python int in the reference and therefore print as "0", not "0.0": the time of row 0 when the path has no
// prologue (motion_profile_generator.py:425), v*12 on every inserted turn / wait row (0 * 12 is the int 0, :448-453,
// 500-503, 511-515), omega on wait rows and on the first row of a turn (:343, :451, :514).
// Pass 1: row text into fixed VAP_ROW_STRIDE-byte slots + lengths.  Pass 2 (after an exclusive scan of the lengths): compact.
#define VAP_ROW_STRIDE 176
#define RK_TIME_INT 1    // times[r] is the int 0 (row 0 of a path whose node 0 has no wait: current_time starts as an int)
#define RK_INSERTED 2    // turn / wait row: linear_vels[r] and accelerations[r] are the int 0
#define RK_OMEGA_INT 4   // angular_vels[r] is the int 0 (wait rows; first row of a turn profile)
#define RK_POS_INT 8     // positions[r] is the int 0 (wait rows)
__global__ void __launch_bounds__(128) k_format_rows(long long R, const double* __restrict__ rows,
                                                     const unsigned char* __restrict__ kinds, char* __restrict__ slots,
                                                     int* __restrict__ lens)
{
    long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    __align__(16) char o[VAP_ROW_STRIDE];          // the line is assembled thread-locally and stored with 16-byte writes
    int n = 0;
    o[n++] = '0'; o[n++] = ' ';
    const double* v = rows + (size_t)r * 7;
    const unsigned kind = kinds ? kinds[r] : 0u;
    for (int c = 1; c < 7; c++) {
        const bool as_int = (c == 1 && (kind & RK_TIME_INT)) || (c == 5 && (kind & RK_INSERTED)) || (c == 6 && (kind & RK_OMEGA_INT));
        if (as_int) { o[n++] = '0'; }
        else n += format_repr(v[c], o + n);
        o[n++] = ' ';
    }
    o[n++] = '\n';
    lens[r] = n;
    uint4* dst = reinterpret_cast<uint4*>(slots + (size_t)r * VAP_ROW_STRIDE);
    const uint4* src = reinterpret_cast<const uint4*>(o);
    for (int k = 0; k < (n + 15) / 16; k++) dst[k] = src[k];
}
__global__ void __launch_bounds__(256) k_compact_rows(long long R, const char* __restrict__ slots, const int* __restrict__ lens,
                                                      const long long* __restrict__ offsets, char* __restrict__ text)
{
    // one warp per row: coalesced byte copies
    long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (r >= R) return;
    const char* s = slots + (size_t)r * VAP_ROW_STRIDE;
    char* d = text + offsets[r];
    int n = lens[r];
    for (int k = lane; k < n; k += 32) d[k] = s[k];
}

// ---- The .txt body of every path: trajectory lines with the action rows spliced in (gui_manager.py:297-310) ----------
// The reference starts from the path's trajectory lines and calls list.insert(nodes_map[i] + i, row) for the node rows,
// then list.insert(actions_map[j] + j, row) for the action-point rows.  Inserted row j ends at a final position P_j; with
// the P_j sorted, Q_j = P_j - j never decreases and trajectory line k has exactly #{j : Q_j <= k} inserted rows in front
// of it.  So one warp per path replays the <= N_max + 1 + A_max inserts on the positions alone (shared memory), ranks
// them, and writes the byte position of every inserted row and every trajectory line; k_compact_rows and
// k_splice_actions then copy the bytes.  Action rows of path b: act_first[b] .. + act_rows[b][0] node rows, then
// act_rows[b][1] action-point rows; row i is act_text[act_off[i] .. act_off[i+1]).
#define SPLICE_OK 0
#define SPLICE_FAILED 1       // status != 0: no action rows (and no lines from vap_export_rows: zero bytes)
#define SPLICE_SHORT 2        // the maps need more action rows than were passed: the body holds the trajectory lines only

// bytes of path b's body and its flag
__device__ __forceinline__ long long splice_path_bytes(long long b, int N_max, int A_stride, const int* __restrict__ status,
                                                       const int* __restrict__ n_maps, const long long* __restrict__ row_off,
                                                       const long long* __restrict__ line_off,
                                                       const long long* __restrict__ act_first, const int* __restrict__ act_rows,
                                                       long long n_act, const long long* __restrict__ act_off, int& flag)
{
    const long long lines = line_off[row_off[b + 1]] - line_off[row_off[b]];
    if (status[b] != 0) { flag = SPLICE_FAILED; return lines; }   // vap_export_rows gives such a path no lines
    const int nm = n_maps[2 * b], am = n_maps[2 * b + 1];
    const long long n0 = act_rows[2 * b], n1 = act_rows[2 * b + 1], a0 = act_first[b];
    if (nm < 0 || am < 0 || nm > N_max + 1 || am > A_stride || n0 < 0 || n1 < 0 || nm > n0 || am > n1 || a0 < 0 ||
        a0 + n0 + n1 > n_act) { flag = SPLICE_SHORT; return lines; }
    flag = SPLICE_OK;
    return lines + (act_off[a0 + nm] - act_off[a0]) + (act_off[a0 + n0 + am] - act_off[a0 + n0]);
}

// path_offsets[B+1] = exclusive scan of the body sizes (one block, as k_row_offsets), flags[B]
__global__ void __launch_bounds__(1024) k_splice_offsets(long long B, int N_max, int A_stride, const int* __restrict__ status,
                                                         const int* __restrict__ n_maps, const long long* __restrict__ row_off,
                                                         const long long* __restrict__ line_off,
                                                         const long long* __restrict__ act_first,
                                                         const int* __restrict__ act_rows, long long n_act,
                                                         const long long* __restrict__ act_off,
                                                         long long* __restrict__ path_off, int* __restrict__ flags)
{
    __shared__ long long s_part[1024];
    const int t = threadIdx.x, NT = blockDim.x;
    const long long per = (B + NT - 1) / NT;
    const long long lo = (long long)t * per, hi = (lo + per < B) ? lo + per : B;
    long long sum = 0;
    int f;
    for (long long b = lo; b < hi; b++)
        sum += splice_path_bytes(b, N_max, A_stride, status, n_maps, row_off, line_off, act_first, act_rows, n_act, act_off, f);
    s_part[t] = sum;
    __syncthreads();
    if (t == 0) {
        long long acc = 0;
        for (int k = 0; k < NT; k++) { long long v = s_part[k]; s_part[k] = acc; acc += v; }
        path_off[B] = acc;
    }
    __syncthreads();
    long long acc = s_part[t];
    for (long long b = lo; b < hi; b++) {
        path_off[b] = acc;
        acc += splice_path_bytes(b, N_max, A_stride, status, n_maps, row_off, line_off, act_first, act_rows, n_act, act_off, f);
        flags[b] = f;
    }
}

// One warp per path.  Shared memory per warp: four arrays of M_cap = N_max + 1 + A_stride entries.
__global__ void __launch_bounds__(128) k_splice_plan(long long B, int N_max, int A_stride, const int* __restrict__ nodes_map,
                                                     const int* __restrict__ actions_map, const int* __restrict__ n_maps,
                                                     const long long* __restrict__ row_off, const long long* __restrict__ line_off,
                                                     const long long* __restrict__ act_first, const int* __restrict__ act_rows,
                                                     const long long* __restrict__ act_off, const long long* __restrict__ path_off,
                                                     const int* __restrict__ flags, long long* __restrict__ line_dst,
                                                     long long* __restrict__ act_dst)
{
    extern __shared__ long long s_splice[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + w;
    if (b >= B) return;
    const int M_cap = N_max + 1 + A_stride;
    long long* pos = s_splice + (size_t)w * 4 * M_cap;    // final position of inserted row j (insert order)
    long long* len = pos + M_cap;                          // its bytes
    long long* sQ = len + M_cap;                           // Q of the inserted rows in final order
    long long* sC = sQ + M_cap;                            // inclusive byte sum of the inserted rows in final order
    const long long r0 = row_off[b], n_lines = row_off[b + 1] - r0, L0 = line_off[r0], base = path_off[b];
    const int flag = flags[b];
    if (flag != SPLICE_OK) {                               // status != 0 has no lines; a short path keeps its lines only
        for (long long k = lane; k < n_lines; k += 32) line_dst[r0 + k] = base + line_off[r0 + k] - L0;
        return;
    }
    const int nm = n_maps[2 * b], am = n_maps[2 * b + 1], M = nm + am;
    const long long a0 = act_first[b], ap0 = a0 + act_rows[2 * b];
    const int* nmap = nodes_map + (size_t)b * (N_max + 1);
    const int* amap = actions_map + (size_t)b * A_stride;
    for (int j = lane; j < M; j += 32) {
        const long long ri = j < nm ? a0 + j : ap0 + (j - nm);
        len[j] = act_off[ri + 1] - act_off[ri];
    }
    for (int j = 0; j < M; j++) {                          // list.insert(idx, row) on a list of n_lines + j entries
        long long idx = j < nm ? (long long)nmap[j] + j : (long long)amap[j - nm] + (j - nm);
        const long long cur = n_lines + j;
        if (idx < 0) { idx += cur; if (idx < 0) idx = 0; }
        if (idx > cur) idx = cur;
        for (int i = lane; i < j; i += 32) if (pos[i] >= idx) pos[i]++;
        __syncwarp();
        if (lane == 0) pos[j] = idx;
        __syncwarp();
    }
    for (int j = lane; j < M; j += 32) {
        const long long p = pos[j];
        long long rank = 0, before = 0;
        for (int i = 0; i < M; i++) if (pos[i] < p) { rank++; before += len[i]; }
        const long long q = p - rank;                      // trajectory lines in front of the row
        const long long ri = j < nm ? a0 + j : ap0 + (j - nm);
        act_dst[ri] = base + (line_off[r0 + q] - L0) + before;
        sQ[rank] = q;
        sC[rank] = before + len[j];
    }
    __syncwarp();
    for (long long k = lane; k < n_lines; k += 32) {
        int lo = 0, hi = M;                                // first rank with Q > k
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (sQ[mid] <= k) lo = mid + 1; else hi = mid; }
        line_dst[r0 + k] = base + (line_off[r0 + k] - L0) + (lo > 0 ? sC[lo - 1] : 0);
    }
}

// the inserted rows into their gaps (one warp per row; rows with act_dst < 0 are not part of any body)
__global__ void __launch_bounds__(256) k_splice_actions(long long n_act, const char* __restrict__ act_text,
                                                        const long long* __restrict__ act_off,
                                                        const long long* __restrict__ act_dst, char* __restrict__ text)
{
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= n_act) return;
    const long long d = act_dst[i];
    if (d < 0) return;
    const char* s = act_text + act_off[i];
    const long long n = act_off[i + 1] - act_off[i];
    for (long long k = lane; k < n; k += 32) text[d + k] = s[k];
}
#endif  // VAP_FORMAT_HOST_TEST
