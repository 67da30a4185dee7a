#include "plan.h"

#include <cmath>
#include <cstdlib>
#include <cstring>

namespace tsnap {

static const size_t kDtypeSize[TSNAP_DTYPE_COUNT] = {1, 1, 2, 4, 8, 2, 2, 4, 8, 1, 1, 1};

size_t dtype_size(int dt) {
    if (dt < 0 || dt >= TSNAP_DTYPE_COUNT) return 0;
    return kDtypeSize[dt];
}

static bool is_float(int dt) { return dt == TSNAP_F16 || dt == TSNAP_BF16 || dt == TSNAP_F32 || dt == TSNAP_F64; }

static bool is_quant(int dt) { return dt == TSNAP_QINT8 || dt == TSNAP_QUINT8; }

bool cast_supported(int s, int d) {
    if (s == d) return !is_quant(s);  // quantised wire elements only exist as the product of a quantising save
    return is_float(s) && (is_float(d) || is_quant(d));
}

static inline uint64_t lowbit(uint64_t x) { return x & (~x + 1); }

// TSNAP_B200_ROWS_MIN_RUN: shortest contiguous run (bytes) that is handed to the copy engine run by run (A/B knob)
static uint64_t rows_min_run() {
    static const uint64_t v = [] {
        const char* e = getenv("TSNAP_B200_ROWS_MIN_RUN");
        const long long x = e ? atoll(e) : 0;
        return x >= 16 ? uint64_t(x) : kRowsMinRun;
    }();
    return v;
}

struct Dim {
    int64_t size, ss, ds;  // strides in bytes
};

static bool tile_fits_u32(const Member& m, int a, int b, uint32_t esz) {
    const uint32_t sa = transpose_side_a(esz), sb = transpose_side_b(esz);
    long double n = 1;
    for (uint32_t i = 0; i < m.nouter; ++i)
        n *= int(i) == a ? (long double)((uint64_t(m.osize[i]) + sa - 1) / sa) : int(i) == b ? (long double)((uint64_t(m.osize[i]) + sb - 1) / sb) : (long double)m.osize[i];
    return n < 4.0e9L;
}

int normalize_copy(const tsnap_copy_desc& d, uint64_t wire_base, bool allow_bulk, NormalizedCopy* out,
                   std::string* err) {
    out->n = 0;
    out->src_space = d.src_space;
    out->dst_space = d.dst_space;
    auto fail = [&](int code, const std::string& msg) {
        if (err) *err = msg;
        return code;
    };
    if (d.ndim < 0 || d.ndim > TSNAP_MAX_DIMS) return fail(TSNAP_EINVAL, "ndim out of range");
    const size_t es = dtype_size(d.src_dtype), ed = dtype_size(d.dst_dtype);
    if (es == 0 || ed == 0) return fail(TSNAP_EINVAL, "unknown dtype");
    if (d.src_space < 0 || d.src_space > TSNAP_SPACE_WIRE || d.dst_space < 0 || d.dst_space > TSNAP_SPACE_WIRE)
        return fail(TSNAP_EINVAL, "unknown address space");
    if (d.src_space == TSNAP_SPACE_WIRE && d.dst_space == TSNAP_SPACE_WIRE)
        return fail(TSNAP_EINVAL, "wire-to-wire copies are not a thing");
    const bool cast = d.src_dtype != d.dst_dtype;
    if (!cast_supported(d.src_dtype, d.dst_dtype))
        return fail(TSNAP_EUNSUP, "unsupported dtype conversion");
    const bool quant = is_quant(d.dst_dtype);
    if (quant && (d.dst_space != TSNAP_SPACE_WIRE || !(d.q_scale > 0)))
        return fail(TSNAP_EINVAL, "quantising copies need a WIRE destination and q_scale > 0");

    // logical shape; C-contiguous element strides for a WIRE destination
    int64_t cstride[TSNAP_MAX_DIMS];
    {
        int64_t acc = 1;
        for (int i = d.ndim - 1; i >= 0; --i) {
            if (d.sizes[i] < 0) return fail(TSNAP_EINVAL, "negative size");
            cstride[i] = acc;
            acc *= d.sizes[i];
        }
    }
    uint64_t numel = 1;
    for (int i = 0; i < d.ndim; ++i) numel *= uint64_t(d.sizes[i]);
    if (numel == 0) return TSNAP_OK;

    Dim dims[TSNAP_MAX_DIMS];
    int nd = 0;
    for (int i = 0; i < d.ndim; ++i) {
        if (d.sizes[i] == 1) continue;
        Dim x;
        x.size = d.sizes[i];
        int64_t ss = d.src_strides[i];
        int64_t ds = d.dst_space == TSNAP_SPACE_WIRE ? cstride[i] : d.dst_strides[i];
        if (ss < 0 || ds < 0) return fail(TSNAP_EINVAL, "negative strides are not supported");
        if (ds == 0) return fail(TSNAP_EINVAL, "destination stride 0 with size > 1 (overlapping writes)");
        x.ss = ss * int64_t(es);
        x.ds = ds * int64_t(ed);
        // merge with the previous (outer) dim when both sides are dense across the boundary
        if (nd > 0 && dims[nd - 1].ss == x.ss * x.size && dims[nd - 1].ds == x.ds * x.size) {
            dims[nd - 1].size *= x.size;
            dims[nd - 1].ss = x.ss;
            dims[nd - 1].ds = x.ds;
        } else {
            dims[nd++] = x;
        }
    }

    Member m;
    std::memset(&m, 0, sizeof(m));
    m.src = d.src_addr + (d.src_space == TSNAP_SPACE_WIRE ? wire_base : 0);
    m.dst = d.dst_addr + (d.dst_space == TSNAP_SPACE_WIRE ? wire_base : 0);
    m.src_dtype = uint32_t(d.src_dtype);
    m.dst_dtype = uint32_t(d.dst_dtype);
    m.src_esz = uint32_t(es);
    m.dst_esz = uint32_t(ed);
    m.bytes = numel * ed;

    if (cast) {
        m.mode = kModeCast;
        m.unit = uint32_t(ed);
        if (quant) {
            m.q_scale = d.q_scale;
            m.q_zero_point = d.q_zero_point;
            m.shift = 1;  // append [scale][zero_point] behind the payload
        }
        if (nd > 0 && dims[nd - 1].ss == int64_t(es) && dims[nd - 1].ds == int64_t(ed)) {
            m.inner = uint64_t(dims[nd - 1].size);
            --nd;
        } else {
            m.inner = 1;
        }
        // the source may be element-misaligned (a wire piece behind an odd-sized slab member): tile_cast then
        // assembles each element from bytes, host_copy_range reads through memcpy
    } else {
        if (nd > 0 && dims[nd - 1].ss == int64_t(es) && dims[nd - 1].ds == int64_t(ed)) {
            m.inner = uint64_t(dims[nd - 1].size) * ed;
            --nd;
        } else {
            m.inner = ed;
        }
    }
    if (nd > kMaxOuter) return fail(TSNAP_EUNSUP, "too many non-mergeable dimensions");
    m.nouter = uint32_t(nd);
    for (int i = 0; i < nd; ++i) {
        m.osize[i] = dims[i].size;
        m.sstride[i] = dims[i].ss;
        m.dstride[i] = dims[i].ds;
    }

    if (cast) {
        out->m[0] = m;
        out->n = 1;
        return TSNAP_OK;
    }
    if (nd == 0) {
        // one dense run on both sides
        const bool device_copy = d.src_space != TSNAP_SPACE_HOST && d.dst_space != TSNAP_SPACE_HOST;
        if (allow_bulk && device_copy && (m.src & 15) == 0 && (m.dst & 15) == 0 && m.bytes >= kBulkMin) {
            const uint64_t body = m.bytes & ~uint64_t(15);
            Member b = m;
            b.mode = kModeBulk;
            b.bytes = body;
            b.inner = body;
            b.unit = 16;
            out->m[out->n++] = b;
            if (m.bytes != body) {
                Member t = m;
                t.mode = kModeContig;
                t.src += body;
                t.dst += body;
                t.bytes = m.bytes - body;
                t.inner = t.bytes;
                t.shift = uint32_t(t.dst & 15);
                t.unit = 1;
                out->m[out->n++] = t;
            }
            return TSNAP_OK;
        }
        m.mode = kModeContig;
        m.shift = uint32_t(m.dst & 15);
        m.unit = uint32_t(lowbit(16 | ((m.src - m.dst) & 15)));  // widest load granule that is aligned whenever dst is
        out->m[0] = m;
        out->n = 1;
        return TSNAP_OK;
    }
    if (m.inner == ed && nd >= 2 && nd <= kMaxOuter) {
        // No run is contiguous on both sides.  If the source is unit-stride along one dim and the destination along
        // another (t(), permute of a dense tensor), tile over those two dims through shared memory.
        int a = -1, b = -1;
        for (int i = 0; i < nd; ++i) {
            if (m.sstride[i] == int64_t(es) && a < 0) a = i;
            if (m.dstride[i] == int64_t(ed) && b < 0) b = i;
        }
        bool aligned = (m.src % es) == 0 && (m.dst % ed) == 0;
        for (int i = 0; i < nd; ++i) aligned = aligned && (uint64_t(m.sstride[i]) % es) == 0 && (uint64_t(m.dstride[i]) % ed) == 0;
        const bool device_copy = d.src_space != TSNAP_SPACE_HOST && d.dst_space != TSNAP_SPACE_HOST;
        if (device_copy && aligned && a >= 0 && b >= 0 && a != b && m.osize[a] >= 16 && m.osize[b] >= 16 && tile_fits_u32(m, a, b, uint32_t(ed))) {
            m.mode = kModeTranspose;
            m.unit = uint32_t(ed);
            m.shift = uint32_t(a) | (uint32_t(b) << 8);
            out->m[0] = m;
            out->n = 1;
            return TSNAP_OK;
        }
    }
    m.mode = kModeStrided;
    uint64_t bits = 16 | m.inner | m.src | m.dst;
    for (int i = 0; i < nd; ++i) bits |= uint64_t(m.sstride[i]) | uint64_t(m.dstride[i]);
    m.unit = uint32_t(lowbit(bits));
    {
        // Column shards / narrow on dim != 0 of wide tables (T:io_preparers/sharded_tensor.py:76, torchrec COLUMN_WISE)
        // and reshard boxes have long 16 B-aligned runs: those go to the copy engine run by run.
        const bool device_copy = d.src_space != TSNAP_SPACE_HOST && d.dst_space != TSNAP_SPACE_HOST;
        if (allow_bulk && device_copy && m.unit == 16 && m.inner >= rows_min_run()) {
            m.mode = kModeRows;
            // is a side laid out run after run (the wire side always is)?
            uint64_t accs = m.inner, accd = m.inner;
            bool sd = true, dd = true;
            for (int i = nd - 1; i >= 0; --i) {
                sd = sd && uint64_t(m.sstride[i]) == accs;
                dd = dd && uint64_t(m.dstride[i]) == accd;
                accs *= uint64_t(m.osize[i]);
                accd *= uint64_t(m.osize[i]);
            }
            m.shift = (sd ? kRowsSrcDense : 0) | (dd ? kRowsDstDense : 0);
        }
    }
    out->m[0] = m;
    out->n = 1;
    return TSNAP_OK;
}

// ---- host execution -------------------------------------------------------------------------------------

static inline float bf16_to_f32(uint16_t v) {
    uint32_t u = uint32_t(v) << 16;
    float f;
    std::memcpy(&f, &u, 4);
    return f;
}
// round-to-nearest-even, NaN -> 0x7FC0: what torch's CPU path produces (c10::BFloat16)
static inline uint16_t f32_to_bf16(float f) {
    if (std::isnan(f)) return 0x7FC0;
    uint32_t u;
    std::memcpy(&u, &f, 4);
    uint32_t bias = ((u >> 16) & 1) + 0x7FFFu;
    return uint16_t((u + bias) >> 16);
}

static inline double load_as_double(const void* p, uint32_t dt) {
    switch (dt) {
        case TSNAP_F16: { _Float16 h; std::memcpy(&h, p, 2); return double(float(h)); }
        case TSNAP_BF16: { uint16_t v; std::memcpy(&v, p, 2); return double(bf16_to_f32(v)); }
        case TSNAP_F32: { float f; std::memcpy(&f, p, 4); return double(f); }
        default: { double x; std::memcpy(&x, p, 8); return x; }
    }
}
// torch's CPU quantisation (FBGEMM's scalar Quantize): zero_point + nearbyint(value * (1.0f / scale)) in float,
// clamped in floating point before the conversion to an integer: a rounded value beyond the int64 range (inf, 1e30)
// has no integer conversion and must saturate at the matching end of the range
static inline uint8_t quantize_host(float x, double scale, int64_t zp, bool is_signed) {
    const float inv = 1.0f / float(scale);
    double q = double(zp) + double(std::nearbyint(x * inv));
    const double lo = is_signed ? -128.0 : 0.0, hi = is_signed ? 127.0 : 255.0;
    q = q > lo ? q : lo;  // also maps NaN to lo instead of an undefined conversion
    q = q < hi ? q : hi;
    return uint8_t(int8_t(int(q)));
}

static inline void store_from(void* p, uint32_t dt, const void* sp, uint32_t sdt) {
    // convert through float when the source is <= 32 bit (exact), through double otherwise.  torch has no direct
    // double -> half conversion: an fp64 source reaches fp16 (and bf16) through fp32, rounded twice, and so does this
    if (sdt == TSNAP_F64) {
        double x;
        std::memcpy(&x, sp, 8);
        switch (dt) {
            case TSNAP_F16: { _Float16 h = (_Float16)float(x); std::memcpy(p, &h, 2); break; }
            case TSNAP_BF16: { uint16_t v = f32_to_bf16(float(x)); std::memcpy(p, &v, 2); break; }
            case TSNAP_F32: { float f = float(x); std::memcpy(p, &f, 4); break; }
            default: std::memcpy(p, &x, 8);
        }
        return;
    }
    float f = float(load_as_double(sp, sdt));
    switch (dt) {
        case TSNAP_F16: { _Float16 h = (_Float16)f; std::memcpy(p, &h, 2); break; }
        case TSNAP_BF16: { uint16_t v = f32_to_bf16(f); std::memcpy(p, &v, 2); break; }
        case TSNAP_F32: std::memcpy(p, &f, 4); break;
        default: { double x = double(f); std::memcpy(p, &x, 8); }
    }
}

static inline void outer_offsets(const Member& m, uint64_t row, int64_t* so, int64_t* dofs) {
    int64_t s = 0, d = 0;
    for (int i = int(m.nouter) - 1; i >= 0; --i) {
        const uint64_t sz = uint64_t(m.osize[i]);
        const uint64_t idx = row % sz;
        row /= sz;
        s += int64_t(idx) * m.sstride[i];
        d += int64_t(idx) * m.dstride[i];
    }
    *so = s;
    *dofs = d;
}

void host_copy_range(const Member& m, uint64_t lo, uint64_t hi) {
    if (hi > m.bytes) hi = m.bytes;
    if (lo >= hi) return;
    const char* src = reinterpret_cast<const char*>(uintptr_t(m.src));
    char* dst = reinterpret_cast<char*>(uintptr_t(m.dst));
    if (m.mode == kModeBulk || m.mode == kModeContig) {
        std::memcpy(dst + lo, src + lo, hi - lo);
        return;
    }
    if (m.mode == kModeStrided || m.mode == kModeRows || m.mode == kModeTranspose) {
        uint64_t pos = lo;
        while (pos < hi) {
            const uint64_t row = pos / m.inner, col = pos % m.inner;
            uint64_t n = m.inner - col;
            if (n > hi - pos) n = hi - pos;
            int64_t so, dofs;
            outer_offsets(m, row, &so, &dofs);
            std::memcpy(dst + dofs + col, src + so + col, n);
            pos += n;
        }
        return;
    }
    // cast: lo/hi are dst bytes, multiples of the dst element size by construction
    const uint64_t e0 = lo / m.dst_esz, e1 = hi / m.dst_esz;
    const bool quant = m.dst_dtype == TSNAP_QINT8 || m.dst_dtype == TSNAP_QUINT8;
    for (uint64_t e = e0; e < e1; ++e) {
        const uint64_t row = e / m.inner, col = e % m.inner;
        int64_t so, dofs;
        outer_offsets(m, row, &so, &dofs);
        if (quant) {
            const float x = float(load_as_double(src + so + col * m.src_esz, m.src_dtype));
            reinterpret_cast<uint8_t*>(dst + dofs)[col] = quantize_host(x, m.q_scale, m.q_zero_point, m.dst_dtype == TSNAP_QINT8);
        } else {
            store_from(dst + dofs + col * m.dst_esz, m.dst_dtype, src + so + col * m.src_esz, m.src_dtype);
        }
    }
    if (quant && (m.shift & 1) && hi == m.bytes) {
        std::memcpy(dst + m.bytes, &m.q_scale, 8);
        std::memcpy(dst + m.bytes + 8, &m.q_zero_point, 8);
    }
}

}  // namespace tsnap
