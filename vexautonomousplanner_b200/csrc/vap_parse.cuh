// vap_parse.cuh -- reading trajectory text back on the device: decimal -> binary64 bit-equal to CPython's float(), the
// lines of concatenated .txt bodies, and the comparison of a saved body against a fresh one.
//
// Token grammar: [-]digits[.digits][e|E[+|-]digits], [-]inf, [-]nan -- everything f"{v}" writes for a trajectory row
// (repr's fixed and exponent forms, -0.0, the int 0 of the RK_* columns), and any other decimal of that form.
// Conversion: the Clinger fast path (w <= 2^53 and |q| <= 22: one correctly rounded multiply or divide), else
// Eisel-Lemire (Lemire, "Number parsing at a gigabyte per second", SPE 2021): the 19 leading significant digits w,
// normalised, times the 128-bit truncated 5^q of vap_pow5_tables.cuh, q in [-342, 308].  A token the algorithm cannot
// decide is not guessed: PARSE_HOST (the caller finishes it with float()) when more than 19 significant digits are
// present and w and w + 1 round differently, or when the 128-bit product is ambiguous (low word all ones outside the
// exact range -27 <= q <= 55).  A token outside the grammar is PARSE_BAD.
#pragma once
#include <cstdint>
#include "vap_pow5_tables.cuh"

#define PARSE_OK 0
#define PARSE_HOST 1          // valid token, not decided on the device: finish it with float()
#define PARSE_BAD 2           // not a token of the grammar

#if defined(__CUDACC__)
#define VAP_HD __host__ __device__
#else
#define VAP_HD
#endif

VAP_HD inline int p_clz64(uint64_t x)
{
#ifdef __CUDA_ARCH__
    return __clzll((long long)x);
#else
    return __builtin_clzll(x);
#endif
}

VAP_HD inline uint64_t p_mulhi(uint64_t a, uint64_t b) { return (uint64_t)(((unsigned __int128)a * b) >> 64); }

VAP_POW5_128_SPACE const double VAP_P10[23] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12,
                                               1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};   // exact

// w * 10^q rounded to nearest even as the IEEE bits of a positive double; false when the product cannot decide it
VAP_HD inline bool eisel_lemire(uint64_t w, int32_t q, uint64_t& bits)
{
    if (w == 0 || q < VAP_POW5_128_QMIN) { bits = 0; return true; }           // below half the least subnormal
    if (q > VAP_POW5_128_QMAX) { bits = 0x7ffull << 52; return true; }        // w >= 1: above the largest double
    const int lz = p_clz64(w);
    w <<= lz;
    const uint64_t* p = VAP_POW5_128[q - VAP_POW5_128_QMIN];
    uint64_t hi = p_mulhi(w, p[0]), lo = w * p[0];
    if ((hi & 0x1ff) == 0x1ff) {                                               // the 9 bits below the 55 kept are all ones
        const uint64_t hi2 = p_mulhi(w, p[1]);
        lo += hi2;
        if (hi2 > lo) hi++;
        if (lo == ~0ull && (q < -27 || q > 55)) return false;
    }
    const int upper = (int)(hi >> 63);
    uint64_t m = hi >> (upper + 9);
    int32_t p2 = (((152170 + 65536) * q) >> 16) + 63 + upper - lz + 1023;
    if (p2 <= 0) {                                                             // subnormal (or rounds up to the least normal)
        if (-p2 + 1 >= 64) { bits = 0; return true; }
        m >>= -p2 + 1;
        m += m & 1;
        m >>= 1;
        bits = m | ((uint64_t)(m < (1ull << 52) ? 0 : 1) << 52);
        return true;
    }
    if (lo <= 1 && q >= -4 && q <= 23 && (m & 3) == 1 && (m << (upper + 9)) == hi) m &= ~1ull;   // exact tie: to even
    m += m & 1;
    m >>= 1;
    if (m >= (2ull << 52)) { m = 1ull << 52; p2++; }
    m &= ~(1ull << 52);
    if (p2 >= 0x7ff) { p2 = 0x7ff; m = 0; }
    bits = ((uint64_t)p2 << 52) | m;
    return true;
}

VAP_HD inline double p_bits_double(uint64_t b)
{
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)b);
#else
    double d;
    __builtin_memcpy(&d, &b, 8);
    return d;
#endif
}

// token s[0 .. n) -> out; returns PARSE_OK / PARSE_HOST / PARSE_BAD (out = NaN unless PARSE_OK)
VAP_HD inline int parse_token(const char* s, long long n, double& out)
{
    out = p_bits_double(0x7ff8000000000000ull);
    long long i = 0;
    const bool neg = n > 0 && s[0] == '-';
    i += neg;
    const uint64_t sign = neg ? (1ull << 63) : 0;
    if (n - i == 3) {
        const char a = s[i], b = s[i + 1], c = s[i + 2];
        if (a == 'i' && b == 'n' && c == 'f') { out = p_bits_double(sign | (0x7ffull << 52)); return PARSE_OK; }
        if (a == 'n' && b == 'a' && c == 'n') { out = p_bits_double(sign | 0x7ff8000000000000ull); return PARSE_OK; }
    }
    uint64_t w = 0;
    int nd = 0;                  // significant digits kept in w (at most 19)
    int32_t q = 0;               // value = w * 10^q (+ the dropped digits)
    bool trunc = false;          // a non-zero digit was dropped
    const long long i0 = i;
    for (; i < n && s[i] >= '0' && s[i] <= '9'; i++) {
        const int d = s[i] - '0';
        if (nd < 19) { w = 10 * w + d; nd += w != 0; }
        else { q += q < 100000; trunc |= d != 0; }
    }
    if (i == i0) return PARSE_BAD;
    if (i < n && s[i] == '.') {
        const long long f0 = ++i;
        for (; i < n && s[i] >= '0' && s[i] <= '9'; i++) {
            const int d = s[i] - '0';
            if (nd < 19) { w = 10 * w + d; nd += w != 0; q -= q > -100000; }
            else trunc |= d != 0;
        }
        if (i == f0) return PARSE_BAD;
    }
    if (i < n && (s[i] == 'e' || s[i] == 'E')) {
        i++;
        bool eneg = false;
        if (i < n && (s[i] == '+' || s[i] == '-')) { eneg = s[i] == '-'; i++; }
        const long long e0 = i;
        int32_t ex = 0;
        for (; i < n && s[i] >= '0' && s[i] <= '9'; i++) if (ex < 100000) ex = 10 * ex + (s[i] - '0');
        if (i == e0) return PARSE_BAD;
        q += eneg ? -ex : ex;
    }
    if (i != n) return PARSE_BAD;
    if (w == 0) { out = p_bits_double(sign); return PARSE_OK; }
    if (!trunc && w <= (1ull << 53) && q >= -22 && q <= 22) {                 // Clinger: both operands exact, one rounding
        const double d = (double)w;
        const double v = q < 0 ? d / VAP_P10[-q] : d * VAP_P10[q];
        out = neg ? -v : v;
        return PARSE_OK;
    }
    uint64_t bits;
    if (!eisel_lemire(w, q, bits)) return PARSE_HOST;
    if (trunc) {                                                               // the true value lies in (w, w + 1) * 10^q
        uint64_t up;
        if (!eisel_lemire(w + 1, q, up) || up != bits) return PARSE_HOST;
    }
    out = p_bits_double(sign | bits);
    return PARSE_OK;
}

#ifndef VAP_PARSE_HOST_TEST
// n tokens text[tok_off[i] .. tok_off[i+1]) -> out[i], flags[i] (PARSE_*)
__global__ void __launch_bounds__(256) k_parse_doubles(long long n, const char* __restrict__ text,
                                                       const long long* __restrict__ tok_off, double* __restrict__ out,
                                                       signed char* __restrict__ flags)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long s = tok_off[i];
    double v;
    flags[i] = (signed char)parse_token(text + s, tok_off[i + 1] - s, v);
    out[i] = v;
}

// ---- Lines of concatenated bodies: body b is text[path_off[b] .. path_off[b+1]); a line ends after '\n' or at the end of
// its body.  Byte i starts a line when it is the first byte of a non-empty body or follows a '\n'.
#define LINE_TRAJ 0           // first token "0": a trajectory row, 7 numeric tokens
#define LINE_ACTION 1         // first token "1": an action row (its tokens stay text)
#define LINE_OTHER 2          // anything else (its error code says what)
#define LINE_ERR_BLANK 1      // no token
#define LINE_ERR_KIND 2       // first token neither 0 nor 1
#define LINE_ERR_TOKENS 3     // trajectory row without exactly 7 tokens
#define LINE_ERR_TOKEN 4      // + column 1..6: a trajectory-row token outside the grammar

__global__ void __launch_bounds__(256) k_line_starts(long long N, const char* __restrict__ text, unsigned char* __restrict__ starts)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    starts[i] = (i == 0 || text[i - 1] == '\n') ? 1 : 0;
}
__global__ void __launch_bounds__(256) k_body_starts(long long B, long long N, const long long* __restrict__ path_off,
                                                     unsigned char* __restrict__ starts)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const long long s = path_off[b];
    if (s < path_off[b + 1] && s < N) starts[s] = 1;
}

// scan[i] = inclusive prefix sum of starts: line k starts at the byte with scan == k + 1 and a start flag
__global__ void __launch_bounds__(256) k_line_offsets(long long N, const unsigned char* __restrict__ starts,
                                                      const int* __restrict__ scan, long long* __restrict__ line_off)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    if (starts[i]) line_off[scan[i] - 1] = i;
}
__global__ void __launch_bounds__(256) k_path_lines(long long B, long long N, const long long* __restrict__ path_off,
                                                    const int* __restrict__ scan, long long* __restrict__ line_off,
                                                    long long* __restrict__ path_line_off)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b > B) return;
    const long long s = path_off[b];
    const long long l = s > 0 ? scan[(s < N ? s : N) - 1] : 0;
    path_line_off[b] = l;
    if (b == B) line_off[l] = N;
}

// kind and first-token error of every line; counts[l] = is trajectory row + 2^32 * is action row (one 1-D scan
// then gives both running counts; each stays below 2^31)
#define CNT_LO(v) ((v) & 0xffffffffLL)
#define CNT_HI(v) ((v) >> 32)
__global__ void __launch_bounds__(256) k_line_kinds(long long L, const char* __restrict__ text, const long long* __restrict__ line_off,
                                                    unsigned char* __restrict__ kinds, int* __restrict__ errors,
                                                    long long* __restrict__ counts)
{
    const long long l = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= L) return;
    const long long s = line_off[l], e = line_off[l + 1];
    long long k = s;
    while (k < e && text[k] != ' ' && text[k] != '\n') k++;
    int kind = LINE_OTHER, err = 0;
    if (k == s) err = LINE_ERR_BLANK;
    else if (k == s + 1 && text[s] == '0') kind = LINE_TRAJ;
    else if (k == s + 1 && text[s] == '1') kind = LINE_ACTION;
    else err = LINE_ERR_KIND;
    kinds[l] = (unsigned char)kind;
    errors[l] = err;
    counts[l] = (long long)(kind == LINE_TRAJ) + ((long long)(kind == LINE_ACTION) << 32);
}

// per body: first trajectory row and first action row (exclusive scans of counts at the body's first line)
__global__ void __launch_bounds__(256) k_path_rows(long long B, const long long* __restrict__ path_line_off,
                                                   const long long* __restrict__ cscan, long long* __restrict__ path_row_off,
                                                   long long* __restrict__ path_act_off)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b > B) return;
    const long long l = path_line_off[b];
    const long long v = l > 0 ? cscan[l - 1] : 0;
    path_row_off[b] = CNT_LO(v);
    path_act_off[b] = CNT_HI(v);
}

// One thread per line.  Action rows: act_line[action index] = line.  Trajectory rows of lines below *n_parse_lines:
// rows[r] = {0, six values}, r = CNT_LO(cscan[l]) - 1; host_mask[l] bit c = column c left for float(); errors as LINE_ERR_*.
__global__ void __launch_bounds__(128) k_parse_lines(long long L, const char* __restrict__ text, const long long* __restrict__ line_off,
                                                     const unsigned char* __restrict__ kinds, const long long* __restrict__ cscan,
                                                     const long long* __restrict__ n_parse_lines, long long* __restrict__ act_line,
                                                     double* __restrict__ rows, unsigned char* __restrict__ host_mask,
                                                     int* __restrict__ errors)
{
    const long long l = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= L) return;
    const int kind = kinds[l];
    if (kind == LINE_ACTION) { act_line[CNT_HI(cscan[l]) - 1] = l; return; }
    if (kind != LINE_TRAJ || l >= *n_parse_lines) return;
    const long long e = line_off[l + 1];
    long long k = line_off[l] + 1;                      // past the first token "0"
    double* row = rows + (size_t)(CNT_LO(cscan[l]) - 1) * 7;
    row[0] = 0.0;
    int ntok = 1, err = 0;
    unsigned mask = 0;
    for (;;) {
        while (k < e && text[k] == ' ') k++;
        if (k >= e || text[k] == '\n') break;
        const long long t0 = k;
        while (k < e && text[k] != ' ' && text[k] != '\n') k++;
        if (ntok < 7) {
            double v;
            const int f = parse_token(text + t0, k - t0, v);
            row[ntok] = v;
            if (f == PARSE_HOST) mask |= 1u << ntok;
            else if (f == PARSE_BAD && err == 0) err = LINE_ERR_TOKEN + ntok;
        }
        ntok++;
    }
    for (int c = ntok; c < 7; c++) row[c] = p_bits_double(0x7ff8000000000000ull);
    if (ntok != 7) err = LINE_ERR_TOKENS;
    host_mask[l] = (unsigned char)mask;
    errors[l] = err;
}

// ---- One saved body against the fresh one, one warp per path ---------------------------------------------------------
#define CMP_DIFF_BYTE 0       // first differing byte from the body start, -1 when the bodies are equal
#define CMP_DIFF_LINE 1       // its line in the saved body, from 1 (0: equal)
#define CMP_OLD_ROWS 2
#define CMP_NEW_ROWS 3
#define CMP_ACTION_DIFF 4     // action rows that differ, the k-th saved one against the k-th fresh one (unpaired ones count)
#define CMP_ERR_LINE 5        // first line of the saved body with an error, from 1 (0: none)
#define CMP_ERR_CODE 6        // its LINE_ERR_* code
#define CMP_NI 7
#define CMP_OLD_T 0           // t of the last trajectory row (NaN without rows)
#define CMP_NEW_T 1
#define CMP_MAXD 2            // + column - 1: max |old - new| of columns 1..6 over the common rows
#define CMP_NF 8

__device__ __forceinline__ long long warp_min_ll(long long v)
{
    for (int o = 16; o > 0; o >>= 1) { const long long u = __shfl_xor_sync(0xffffffffu, v, o); v = u < v ? u : v; }
    return v;
}
__device__ __forceinline__ double warp_max_d(double v)
{
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__global__ void __launch_bounds__(128) k_compare_bodies(long long B, const char* __restrict__ text,
                                                        const long long* __restrict__ old_off, const long long* __restrict__ new_off,
                                                        const long long* __restrict__ line_off, const int* __restrict__ line_err,
                                                        const long long* __restrict__ old_pl, const long long* __restrict__ act_line,
                                                        const long long* __restrict__ old_pa, const long long* __restrict__ new_pa,
                                                        const double* __restrict__ old_rows, const long long* __restrict__ old_ro,
                                                        const double* __restrict__ new_rows, const long long* __restrict__ new_ro,
                                                        long long* __restrict__ out_i, double* __restrict__ out_f)
{
    const int lane = threadIdx.x & 31;
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B) return;
    const long long o0 = old_off[b], lo = old_off[b + 1] - o0, n0 = new_off[b], ln = new_off[b + 1] - n0;
    const long long m = lo < ln ? lo : ln;
    const long long NONE = 0x7fffffffffffffffLL;
    long long diff = NONE;
    for (long long base = 0; base < m && diff == NONE; base += 32 * 16) {
        long long mine = NONE;
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const long long i = base + k * 32 + lane;
            if (i < m && mine == NONE && text[o0 + i] != text[n0 + i]) mine = i;
        }
        if (__any_sync(0xffffffffu, mine != NONE)) diff = warp_min_ll(mine);
    }
    if (diff == NONE && lo != ln) diff = m;
    const long long pl0 = old_pl[b], pl1 = old_pl[b + 1];
    long long err_l = NONE;
    for (long long l = pl0 + lane; l < pl1; l += 32) if (line_err[l] != 0) { err_l = l; break; }
    err_l = warp_min_ll(err_l);

    const long long ro0 = old_ro[b], nro = old_ro[b + 1] - ro0, rn0 = new_ro[b], nrn = new_ro[b + 1] - rn0;
    const long long common = nro < nrn ? nro : nrn;
    double md[6] = {0, 0, 0, 0, 0, 0};
    for (long long k = lane; k < common; k += 32) {
        const double* a = old_rows + (size_t)(ro0 + k) * 7;
        const double* c = new_rows + (size_t)(rn0 + k) * 7;
#pragma unroll
        for (int j = 0; j < 6; j++) {
            const double x = a[j + 1], y = c[j + 1];
            double d = (x == y || (x != x && y != y)) ? 0.0 : fabs(x - y);
            if (d != d) d = __longlong_as_double(0x7ff0000000000000LL);
            md[j] = fmax(md[j], d);
        }
    }
#pragma unroll
    for (int j = 0; j < 6; j++) md[j] = warp_max_d(md[j]);

    const long long pa0 = old_pa[b], nao = old_pa[b + 1] - pa0, pn0 = new_pa[b], nan_ = new_pa[b + 1] - pn0;
    const long long acommon = nao < nan_ ? nao : nan_;
    long long adiff = 0;
    for (long long k = lane; k < acommon; k += 32) {
        const long long la = act_line[pa0 + k], lb = act_line[pn0 + k];
        const long long sa = line_off[la], ea = line_off[la + 1], sb = line_off[lb], eb = line_off[lb + 1];
        bool same = ea - sa == eb - sb;
        for (long long i = 0; same && i < ea - sa; i++) same = text[sa + i] == text[sb + i];
        adiff += !same;
    }
    for (int o = 16; o > 0; o >>= 1) adiff += __shfl_xor_sync(0xffffffffu, adiff, o);
    if (lane != 0) return;
    long long dline = 0;
    if (diff != NONE) {
        const long long pos = o0 + diff;
        long long a = pl0, z = pl1;                      // lines of the saved body starting at or before pos
        while (a < z) { const long long mid = (a + z) >> 1; if (line_off[mid] <= pos) a = mid + 1; else z = mid; }
        dline = a - pl0;
        if (diff == lo && (lo == 0 || text[o0 + lo - 1] == '\n')) dline++;    // past the last '\n': a new line
    }
    long long* oi = out_i + (size_t)b * CMP_NI;
    oi[CMP_DIFF_BYTE] = diff == NONE ? -1 : diff;
    oi[CMP_DIFF_LINE] = dline;
    oi[CMP_OLD_ROWS] = nro;
    oi[CMP_NEW_ROWS] = nrn;
    oi[CMP_ACTION_DIFF] = adiff + (nao > nan_ ? nao - nan_ : nan_ - nao);
    oi[CMP_ERR_LINE] = err_l == NONE ? 0 : err_l - pl0 + 1;
    oi[CMP_ERR_CODE] = err_l == NONE ? 0 : line_err[err_l];
    double* of = out_f + (size_t)b * CMP_NF;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    of[CMP_OLD_T] = nro > 0 ? old_rows[(size_t)(ro0 + nro - 1) * 7 + 1] : qnan;
    of[CMP_NEW_T] = nrn > 0 ? new_rows[(size_t)(rn0 + nrn - 1) * 7 + 1] : qnan;
    for (int j = 0; j < 6; j++) of[CMP_MAXD + j] = md[j];
}
#endif  // VAP_PARSE_HOST_TEST
