// Row N8: mixed batches of dataset files, the listing of the reference's evaluation.get_data_list (*.jpg, *.png and
// *.pgm in one dataset), in one call.  Every file is sniffed by its leading bytes (JPEG FF D8 FF, the PNG signature,
// a netpbm magic "Pn") and parsed on the host; the JPEG files go through jpeg.cu's decoder and the PNG files through
// png.cu's, each on its subset, one after the other on the context's stream, and each writes its photos at their
// offsets in one photo buffer; a binary PGM's payload is the photo itself and reaches that buffer by a plain copy.
// Photo preparation (image_prep.cu) then reads colour photos as RGB and gray ones (1-component JPEG, PNG colour types 0
// and 4, PGM) as gray; DESIGN.md section 4.10.
#include <algorithm>
#include "vpk_internal.cuh"

namespace vpk {

static bool pnm_space(uint8_t c) { return c == ' ' || c == '\t' || c == '\n' || c == '\v' || c == '\f' || c == '\r'; }

// the next header number of a netpbm file: whitespace and '#' comments (to the end of the line) skipped, then decimal
// digits; false when there are none or the value exceeds INT32_MAX
static bool pnm_number(const uint8_t* p, int64_t n, int64_t& i, int64_t& v) {
    for (;;) {
        if (i >= n) return false;
        if (pnm_space(p[i])) { ++i; continue; }
        if (p[i] == '#') { while (i < n && p[i] != '\n' && p[i] != '\r') ++i; continue; }
        break;
    }
    if (p[i] < '0' || p[i] > '9') return false;
    v = 0;
    while (i < n && p[i] >= '0' && p[i] <= '9') {
        v = v * 10 + (p[i] - '0');
        if (v > INT32_MAX) return false;
        ++i;
    }
    return true;
}

// A netpbm file (p[0] == 'P', p[1] in '1'..'7'): VPK_PGM_OK for a binary PGM (P5) with maxval 255 and its whole
// payload, else the reason.  w / h are set once the header has them, *payload once maxval and its whitespace byte
// are read.
static int pgm_parse(const uint8_t* p, int64_t n, int32_t& w, int32_t& h, int64_t& payload) {
    w = h = 0;
    payload = 0;
    switch (p[1]) {
        case '2': return VPK_PGM_ASCII;
        case '1': case '4': return VPK_PGM_BITMAP;
        case '3': case '6': return VPK_PGM_PPM;
        case '7': return VPK_PGM_PAM;
        default: break;
    }
    int64_t i = 2, W = 0, H = 0, M = 0;
    if (i >= n || !(pnm_space(p[i]) || p[i] == '#')) return VPK_PGM_MALFORMED;
    if (!pnm_number(p, n, i, W) || !pnm_number(p, n, i, H) || W <= 0 || H <= 0) return VPK_PGM_MALFORMED;
    w = (int32_t)W; h = (int32_t)H;
    if (!pnm_number(p, n, i, M) || M <= 0 || M > 65535) return VPK_PGM_MALFORMED;
    if (i >= n || !pnm_space(p[i])) return VPK_PGM_MALFORMED;      // exactly one whitespace byte before the payload
    payload = i + 1;
    if (M > 255) return VPK_PGM_DEPTH;
    if (M < 255) return VPK_PGM_MAXVAL;
    if (n - payload < W * H) return VPK_PGM_MALFORMED;               // truncated; extra bytes after it are allowed
    return VPK_PGM_OK;
}

static const char* pgm_reason_name(int r) {
    switch (r) {
        case VPK_PGM_ASCII: return "ASCII PGM (P2)";
        case VPK_PGM_BITMAP: return "bitmap (P1 / P4)";
        case VPK_PGM_PAM: return "PAM (P7)";
        case VPK_PGM_PPM: return "PPM (P3 / P6)";
        case VPK_PGM_MAXVAL: return "maxval below 255";
        case VPK_PGM_DEPTH: return "16-bit samples (maxval above 255)";
        case VPK_PGM_MALFORMED: return "malformed header or truncated payload";
        default: return "unknown";
    }
}

static const char* format_name(int f) {
    switch (f) {
        case VPK_FILE_JPEG: return "JPEG";
        case VPK_FILE_PNG: return "PNG";
        case VPK_FILE_PGM: return "PGM";
        default: return "unknown format";
    }
}

static int sniff(const uint8_t* p, int64_t n) {
    if (n >= 3 && p[0] == 0xFF && p[1] == 0xD8 && p[2] == 0xFF) return VPK_FILE_JPEG;
    if (n >= 8 && memcmp(p, "\x89PNG\r\n\x1a\n", 8) == 0) return VPK_FILE_PNG;
    if (n >= 2 && p[0] == 'P' && p[1] >= '1' && p[1] <= '7') return VPK_FILE_PGM;
    return VPK_FILE_UNKNOWN;
}

struct FileInfo {
    int32_t fmt = VPK_FILE_UNKNOWN, w = 0, h = 0, c = 0, support = 1;
    int64_t payload = 0;        // PGM: offset of the payload in the file
};

// one file's format, size, channels of its decoded photo and support (the format's own reason code; 1 if unknown)
static void file_info(const uint8_t* p, int64_t n, FileInfo& f) {
    f = FileInfo();
    f.fmt = sniff(p, n);
    const int64_t off[2] = {0, n};
    if (f.fmt == VPK_FILE_JPEG) {
        vpk_jpeg_info(p, off, 1, &f.w, &f.h, &f.c, &f.support);
    } else if (f.fmt == VPK_FILE_PNG) {
        int32_t ctype = 0;
        vpk_png_info(p, off, 1, &f.w, &f.h, &ctype, &f.support);
        f.c = f.w > 0 ? (ctype == 0 || ctype == 4 ? 1 : 3) : 0;
    } else if (f.fmt == VPK_FILE_PGM) {
        f.support = pgm_parse(p, n, f.w, f.h, f.payload);
        f.c = f.w > 0 ? 1 : 0;
    }
}

static int check_offsets(const uint8_t* data, const int64_t* byte_offsets, int32_t B, const char* who) {
    if (!byte_offsets || B <= 0) { set_error("%s: bad argument", who); return VPK_ERR_ARG; }
    for (int b = 0; b < B; ++b)
        if (byte_offsets[b + 1] < byte_offsets[b] || byte_offsets[b] < 0) { set_error("%s: byte_offsets must be non-decreasing from >= 0", who); return VPK_ERR_ARG; }
    if (!data && byte_offsets[B] > byte_offsets[0]) { set_error("%s: data is NULL", who); return VPK_ERR_ARG; }
    return VPK_OK;
}

int files_plan(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t B, const char* who, FilesPlan& p) {
    VPK_TRY(check_offsets(data, byte_offsets, B, who));
    p = FilesPlan();
    p.B = B; p.data = data; p.byte_offsets = byte_offsets;
    p.fmt.resize(B); p.w.resize(B); p.h.resize(B); p.c.resize(B);
    p.pix_off.assign(B + 1, 0);
    for (int b = 0; b < B; ++b) {
        FileInfo f;
        file_info(data + byte_offsets[b], byte_offsets[b + 1] - byte_offsets[b], f);
        if (f.fmt == VPK_FILE_UNKNOWN) {
            set_error("%s: file %d is not supported: unknown format (not JPEG, PNG or PGM)", who, b);
            return VPK_ERR_ARG;
        }
        if (f.support != 0) {
            const char* why = f.fmt == VPK_FILE_JPEG ? jpeg_reason_name(f.support) : f.fmt == VPK_FILE_PNG ? png_reason_name(f.support)
                                                                                                             : pgm_reason_name(f.support);
            set_error("%s: file %d (%s) is not supported: reason %d (%s)", who, b, format_name(f.fmt), f.support, why);
            return VPK_ERR_ARG;
        }
        p.fmt[b] = f.fmt; p.w[b] = f.w; p.h[b] = f.h; p.c[b] = f.c;
        p.pix_off[b + 1] = p.pix_off[b] + (int64_t)f.c * f.w * f.h;
        if (f.fmt == VPK_FILE_PGM) {
            p.pgm.push_back(b);
            p.pgm_payload.push_back(byte_offsets[b] + f.payload);
        } else {
            p.sub[f.fmt == VPK_FILE_JPEG ? 0 : 1].push_back(b);
        }
    }
    // each decoder reads its files from one range with cumulative offsets: the caller's bytes when its files are
    // consecutive there (a batch of one format), else a host pack of them
    for (int k = 0; k < 2; ++k) {
        const std::vector<int32_t>& s = p.sub[k];
        const int n = (int)s.size();
        if (!n) continue;
        bool contiguous = true;
        for (int j = 0; j + 1 < n && contiguous; ++j) contiguous = byte_offsets[s[j] + 1] == byte_offsets[s[j + 1]];
        std::vector<int64_t>& off = p.sub_off[k];
        off.assign(n + 1, 0);
        if (contiguous) {
            const int64_t base = byte_offsets[s[0]];
            for (int j = 0; j < n; ++j) off[j + 1] = byte_offsets[s[j] + 1] - base;
            p.sub_data[k] = data + base;
        } else {
            for (int j = 0; j < n; ++j) off[j + 1] = off[j] + byte_offsets[s[j] + 1] - byte_offsets[s[j]];
            p.pack[k].resize((size_t)std::max<int64_t>(off[n], 1));
            for (int j = 0; j < n; ++j)
                if (off[j + 1] > off[j]) memcpy(p.pack[k].data() + off[j], data + byte_offsets[s[j]], (size_t)(off[j + 1] - off[j]));
            p.sub_data[k] = p.pack[k].data();
        }
        std::vector<int32_t> w, h, c;
        if (k == 0) VPK_TRY(jpeg_plan(ctx, p.sub_data[k], off.data(), n, false, who, w, h, c));
        else VPK_TRY(png_plan(ctx, p.sub_data[k], off.data(), n, false, who, w, h, c));
    }
    return VPK_OK;
}

int files_decode(vpk_ctx* ctx, const FilesPlan& p, uint8_t* d_out, int32_t* status_out) {
    VPK_CUDA(cudaSetDevice(ctx->device));
    for (int k = 0; k < 2; ++k) {
        const std::vector<int32_t>& s = p.sub[k];
        const int n = (int)s.size();
        if (!n) continue;
        // the decoders place file j at pix_off[j] and bound their writes by pix_off[n]
        std::vector<int64_t> pix(n + 1);
        for (int j = 0; j < n; ++j) pix[j] = p.pix_off[s[j]];
        pix[n] = p.pix_off[p.B];
        std::vector<int32_t> st(n);
        if (k == 0) VPK_TRY(jpeg_decode(ctx, p.sub_data[k], p.sub_off[k].data(), pix.data(), d_out, st.data()));
        else VPK_TRY(png_decode(ctx, p.sub_data[k], p.sub_off[k].data(), pix.data(), d_out, st.data()));
        for (int j = 0; j < n; ++j) status_out[s[j]] = st[j];
    }
    for (size_t j = 0; j < p.pgm.size(); ++j) {
        const int b = p.pgm[j];
        VPK_CUDA(cudaMemcpyAsync(d_out + p.pix_off[b], p.data + p.pgm_payload[j], (size_t)(p.pix_off[b + 1] - p.pix_off[b]),
                                 cudaMemcpyHostToDevice, ctx->stream));
        status_out[b] = VPK_PGM_OK;
    }
    return VPK_OK;
}

}  // namespace vpk

using namespace vpk;

extern "C" {

int vpk_file_info(const uint8_t* data, const int64_t* byte_offsets, int32_t n, int32_t* formats, int32_t* widths, int32_t* heights,
                  int32_t* channels, int32_t* support) {
    VPK_TRY(check_offsets(data, byte_offsets, n, "vpk_file_info"));
    for (int b = 0; b < n; ++b) {
        FileInfo f;
        file_info(data + byte_offsets[b], byte_offsets[b + 1] - byte_offsets[b], f);
        if (formats) formats[b] = f.fmt;
        if (widths) widths[b] = f.w;
        if (heights) heights[b] = f.h;
        if (channels) channels[b] = f.c;
        if (support) support[b] = f.support;
    }
    return VPK_OK;
}

int vpk_decode_files(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n, uint8_t* pixels_out, int32_t* status_out) {
    if (!ctx || !pixels_out || !status_out) { set_error("vpk_decode_files: bad argument"); return VPK_ERR_ARG; }
    FilesPlan fp;
    VPK_TRY(files_plan(ctx, data, byte_offsets, n, "vpk_decode_files", fp));
    PrepPlan pp;
    VPK_TRY(prep_plan(fp.pix_off.data(), fp.w.data(), fp.h.data(), fp.c.data(), n, 0, "vpk_decode_files", pp));
    uint8_t* d_pix = nullptr;
    VPK_TRY(prep_input(ctx, pp, &d_pix));
    VPK_TRY(files_decode(ctx, fp, d_pix, status_out));
    VPK_CUDA(cudaMemcpyAsync(pixels_out, d_pix, (size_t)fp.pix_off[n], cudaMemcpyDeviceToHost, ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    return VPK_OK;
}

int vpk_prepare_files(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n, int32_t target_size,
                      int32_t* out_widths, int32_t* out_heights, double* planes_out) {
    if (!ctx || !out_widths || !out_heights || !planes_out) { set_error("vpk_prepare_files: bad argument"); return VPK_ERR_ARG; }
    FilesPlan fp;
    VPK_TRY(files_plan(ctx, data, byte_offsets, n, "vpk_prepare_files", fp));
    PrepPlan pp;
    VPK_TRY(prep_plan(fp.pix_off.data(), fp.w.data(), fp.h.data(), fp.c.data(), n, target_size, "vpk_prepare_files", pp));
    VPK_CUDA(cudaSetDevice(ctx->device));
    uint8_t* d_pix = nullptr;
    VPK_TRY(prep_input(ctx, pp, &d_pix));
    std::vector<int32_t> status(n);
    VPK_TRY(files_decode(ctx, fp, d_pix, status.data()));
    const int64_t n_out = pp.pix_off[n];
    double* d_out = nullptr;
    VPK_TRY(prep_output(ctx, n_out, &d_out));
    VPK_TRY(prep_run(ctx, pp, 1.0, d_out));
    VPK_CUDA(cudaMemcpyAsync(planes_out, d_out, (size_t)n_out * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    VPK_CUDA(cudaStreamSynchronize(ctx->stream));
    memcpy(out_widths, pp.W.data(), (size_t)n * sizeof(int32_t));
    memcpy(out_heights, pp.H.data(), (size_t)n * sizeof(int32_t));
    return VPK_OK;
}

}  // extern "C"
