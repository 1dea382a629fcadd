// Streaming objects of the C ABI: afe_mfcc (MfccOpenCL replacement), afe_segmenter, afe_delta, afe_normalizer.
// Host-side state machines follow the reference CPU classes (segmentercpu.cpp:56-106, mfcccpu.cpp:338-444).
// afe_mfcc runs every block through the fused kernel K1 (afe_fused.cuh): ONE launch per apply(), the block being a
// "tile group" with its carried-over context as halo; parameter sets K1 does not cover (other FFT sizes, odd shifts,
// normalisation before the deltas) take the staged kernels of afe_stages.cu. One CUDA stream per object; a verb only
// waits for the device where it hands data back to the host (get_output, like the blocking reads of mfccopencl.cpp:78-90).
#include <algorithm>
#include <cstring>
#include <memory>

#include "afe_internal.h"
#include "afe_fused_host.h"
#include "afe_nccl.h"

using namespace afe;

namespace {

// Carry-over bookkeeping shared by afe_segmenter and afe_mfcc (segmentercpu.cpp). PCM lives on the device in two
// ping-pong buffers: `cur` holds [carry-over | new block]; after the frames are cut the tail is copied to the front
// of the other buffer.
struct SegState {
    int W, S, N2, D, frame_cap;
    int remaining = 0, samples = 0;
    bool flushed = true, last_calc_flushed = false;
    size_t cap = 0;
    DevBuf<int16_t> buf[2];
    // pinned staging (two buffers, alternating) so that the H2D copy is asynchronous and the caller may reuse its buffer
    // at once; a buffer is reused only after the copy that read it has completed (event), which by then it normally has
    PinnedBuf<int16_t> h_pin[2];
    bool pin_busy[2] = {false, false}; // an H2D copy out of this staging buffer may still be running; cleared by synced()
    int cur = 0, pin = 0;
    bool carry_pending = false; // the tail of buf[cur] still has to move to the front of buf[cur ^ 1] (done by the next set_input;
                                // flush() reads the tail where it lies, so a single-block stream never copies it)
    float pre = 0.f;          // pre-emphasis coefficient (staged segmenter path)

    void init(int W_, int S_, int frame_cap_, int D_)
    {
        W = W_; S = S_; D = D_; frame_cap = frame_cap_;
        N2 = afe_fft_size(W);
        cap = (size_t)frame_cap * S + W - S;                 // segmentercpu.cpp:40
        for (auto &b : buf) {
            b.alloc(cap + N2 + 16);                          // + slack: the FFT kernel reads whole N2-sample words
            AFE_CUDA(cudaMemset(b.p, 0, sizeof(int16_t) * (cap + N2 + 16)));
        }
        for (auto &h : h_pin) h.alloc(cap);
    }
    void reset() { remaining = samples = 0; flushed = true; last_calc_flushed = false; carry_pending = false; }
    void synced() { pin_busy[0] = pin_busy[1] = false; } // the owner synchronised the stream: every staged copy has landed
    int est(int n) const { return afe_estimated_window_count(n, W, S); }

    // Returns the device pointer holding this block's contiguous PCM (valid until the next call).
    const int16_t *set_input(const int16_t *in, int n, int &wc, int &wc_nd, cudaStream_t st)
    {
        if ((size_t)n + (flushed ? 0 : remaining) > cap) throw Error("Can't process data, buffer is too small");
        if (!flushed && carry_pending) {                     // carry-over to the front of the other buffer, then append
            const int16_t *src = buf[cur].p + samples - remaining;
            AFE_CUDA(cudaMemcpyAsync(buf[cur ^ 1].p, src, sizeof(int16_t) * remaining, cudaMemcpyDeviceToDevice, st));
            cur ^= 1;
        }
        carry_pending = false;
        int16_t *dst = buf[cur].p;
        int total = n;
        if (flushed) {                                       // first block of a stream (segmentercpu.cpp:59-75)
            total = n;
            wc_nd = est(total);
            wc = wc_nd - D;
            // wc < D would put the carry-over in front of the buffer (the reference reads out of bounds there,
            // segmentercpu.cpp:69-73): same error as for wc <= 0
            if (wc <= 0 || wc < D) throw Error("Can't process data, window count is too small");
            const int used = (wc - D) * S + W - S;
            if (used <= 0) throw Error("Processed samples <= 0, this should never happen");
        }
        last_calc_flushed = flushed;
        pin ^= 1;
        if (pin_busy[pin]) { AFE_CUDA(cudaStreamSynchronize(st)); synced(); } // rare: two blocks without a get_output between
        memcpy(h_pin[pin].p, in, sizeof(int16_t) * n);
        pin_busy[pin] = true;
        if (flushed) {
            AFE_CUDA(cudaMemcpyAsync(dst, h_pin[pin].p, sizeof(int16_t) * n, cudaMemcpyHostToDevice, st));
            const int used = (wc - D) * S + W - S;
            remaining = total - used + W - S;
            flushed = false;
        } else {                                             // append to the carry-over (segmentercpu.cpp:76-93)
            AFE_CUDA(cudaMemcpyAsync(dst + remaining, h_pin[pin].p, sizeof(int16_t) * n, cudaMemcpyHostToDevice, st));
            total = n + remaining;
            wc_nd = est(total);
            wc = wc_nd - 2 * D;
            if (wc < 0) wc = 0;
            const int used = wc * S + W - S;
            remaining = total - used + W - S;
        }
        samples = total;
        return dst;
    }
    // after the frames of the current block were cut: its tail is the next block's head (moved lazily, see carry_pending)
    void carry(cudaStream_t) { carry_pending = true; }
    const int16_t *flush(int &wc, int &wc_nd)                // segmentercpu.cpp:97-106
    {
        flushed = true;
        wc_nd = est(remaining);
        wc = wc_nd - D;
        const int16_t *src = carry_pending ? buf[cur].p + samples - remaining : buf[cur].p;
        carry_pending = false;
        return src;
    }
};

} // namespace

// ================================================================================================== afe_mfcc
struct afe_mfcc {
    Derived d;
    int device;
    Stream st;
    SegState seg;
    float alpha = 1.f, pre = 0.f;
    bool window_set = false, last_block = false, fix_q1 = false;
    std::vector<float> window;
    DevBuf<float> outb;
    PinnedBuf<float> h_out;
    // ---- fused route: every block is ONE launch of K1
    std::unique_ptr<FusedEngine> eng;
    const int16_t *blk_pcm = nullptr;   // device PCM of the current block (carry-over + new samples)
    size_t tiles_cap = 0;
    // Speculative flush rows: every apply() of a non-final block also computes, in the same launch, the D rows a flush()
    // right after it would return (outb rows [wc, wc + D)). flush() -> apply() -> get_output_data() then costs no launch
    // as long as alpha and the Q1 option are still the ones those rows were computed with.
    bool spec_valid = false, spec_fix_q1 = false, out_is_spec = false;
    float spec_alpha = 0.f;
    int spec_row0 = 0;
    bool spec_on_host = false;          // the speculative rows already travelled to h_out with the block's rows
    bool pending = false;               // work enqueued on the stream since the last synchronisation
    FusedNormState norm;                // one group: the block; mean / scale also serve the flush block (use_last_stats)
    int launches = 0;
    // ---- staged route (parameter sets K1 does not cover): one kernel per reference stage, spectrum persisted
    FftTables fft;
    MelTables mel;
    NormState n0, n1, n2;
    DevBuf<float> mag, melv, cep, dpad, d1, d2;
    afe_mfcc(const afe_params &p, int dev) : d(p), device(dev) {}
    bool fused() const { return (bool)eng; }
    float *statics() { return d.C > 0 ? cep.p : melv.p; }
    // Row offset of this block's first OUTPUT static: the reference keys it on was_flushed() (mfcccpu.cpp:274,439),
    // which is still true when flushing after a single set_input (quirk Q1) unless the fix is requested.
    int static_row_offset() const { return (!seg.last_calc_flushed || (fix_q1 && last_block)) ? d.D : 0; }
};

// buffers of the staged route (one kernel per reference stage)
static void alloc_staged(afe_mfcc *h)
{
    const Derived &d = h->d;
    const size_t fc = d.frame_cap;
    if (d.N2 == 512 || d.N2 == 256) h->fft.build(d.N2);
    h->mag.alloc(fc * d.bins);
    h->melv.alloc(fc * d.nb);
    if (d.C > 0) h->cep.alloc(fc * d.dct_len);
    if (d.p.norm != AFE_NORM_NONE) { h->n0.init(d.p.norm, d.cols); h->n1.init(d.p.norm, d.cols); h->n2.init(d.p.norm, d.cols); }
    if (d.p.dyn != AFE_DYN_NONE) {
        h->dpad.alloc((fc + 2 * d.D) * d.cols);          // m_delta_in, mfcccpu.cpp:148-156
        h->d1.alloc((fc + 2 * d.l2) * d.cols);
        h->d2.alloc(fc * d.cols);
    }
}

extern "C" {

int afe_mfcc_create(const afe_params *p, int cuda_device, afe_mfcc **out)
{
    *out = nullptr;
    return guarded([&] {
        if (afe_device_count() <= cuda_device) throw Error("no usable CUDA device " + std::to_string(cuda_device) + " (the product has no CPU fallback)");
        DeviceGuard g(cuda_device);
        std::unique_ptr<afe_mfcc> h(new afe_mfcc(*p, cuda_device));
        const Derived &d = h->d;
        if (d.in_frames_cap < 1) throw Error("input_buffer_size is smaller than one window");
        h->st.create();
        h->seg.init(d.W, d.S, d.frame_cap, d.D);
        const size_t fc = d.frame_cap;
        // K1 covers the block when the parameter set fits it and normalisation (if any) comes after the deltas: normalising
        // BEFORE them takes statistics over the look-ahead rows of the block as well (mfcccpu.cpp:383-384), which no tile owns
        // (1024-point FFTs stay on the staged kernels here: K1 serves them in the batch extractor only)
        const bool fused = fused_unsupported_reason(d).empty() && d.N2 <= 512 && (d.p.norm == AFE_NORM_NONE || d.p.norm_after_dyn);
        if (fused) {
            h->eng.reset(new FusedEngine(d, cuda_device));
            h->tiles_cap = fc / 32 + 2 * (size_t)h->eng->sm_count + 8;
            if (d.p.norm != AFE_NORM_NONE) h->norm.alloc(1, h->tiles_cap + 1, d.width);
        } else
            alloc_staged(h.get());
        h->outb.alloc((fc + d.D) * d.width);
        h->h_out.alloc((fc + d.D) * d.width);
        *out = h.release();
    });
}

void afe_mfcc_destroy(afe_mfcc *h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->st);
    delete h;
}

int afe_mfcc_set_window(afe_mfcc *h, const float *window)
{
    return guarded([&] {
        DeviceGuard g(h->device);
        if (h->fused()) h->eng->set_window(window, h->st);
        else upload_window(h->d, window, h->mel, h->st);
        h->window_set = true;
    });
}
int afe_mfcc_set_alpha(afe_mfcc *h, float alpha) { h->alpha = alpha; return 0; }
int afe_mfcc_set_preemphasis(afe_mfcc *h, float coefficient)
{
    return guarded([&] {
        if (!(coefficient >= 0.f && coefficient < 1.f)) throw Error("pre-emphasis coefficient must be in [0, 1)");
        h->pre = coefficient;
        if (h->fused()) h->eng->pre = coefficient;
    });
}
int afe_mfcc_input_buffer_size(const afe_mfcc *h) { return h->d.in_cap; }
int afe_mfcc_estimated_window_count(const afe_mfcc *h, int samples) { return afe_estimated_window_count(samples, h->d.W, h->d.S); }
int afe_mfcc_output_width(const afe_mfcc *h) { return h->d.width; }
int afe_mfcc_uses_fused_kernel(const afe_mfcc *h) { return h->fused() ? 1 : 0; }
int afe_mfcc_kernel_launches(const afe_mfcc *h) { return h->launches; }
int afe_mfcc_set_option(afe_mfcc *h, int option, int value)
{
    if (option == AFE_OPT_FIX_FLUSH_STATICS) { h->fix_q1 = value != 0; return 0; }
    if (option == AFE_OPT_STAGED_KERNELS) {
        // A-B switch: run the blocks through the staged kernels although the fused kernel covers the parameter set
        return guarded([&] {
            if (h->window_set) throw Error("AFE_OPT_STAGED_KERNELS must be set before set_window");
            if (value != 0 && h->fused()) { DeviceGuard g(h->device); h->eng.reset(); alloc_staged(h); }
            else if (value == 0 && !h->fused()) throw Error("the staged kernels cannot be switched off for this parameter set");
        });
    }
    return fail("unknown option");
}
int afe_mfcc_reset(afe_mfcc *h)
{
    return guarded([&] {
        DeviceGuard g(h->device);
        if (h->pending) { AFE_CUDA(cudaStreamSynchronize(h->st)); h->pending = false; h->seg.synced(); }
        h->seg.reset(); h->last_block = false; h->spec_valid = false; h->out_is_spec = false; h->spec_on_host = false;
    });
}

int afe_mfcc_set_input(afe_mfcc *h, const int16_t *data, int samples, int *frames)
{
    *frames = 0;
    return guarded([&] {
        if (!h->window_set) throw Error("set_window must be called before set_input");
        if (samples > h->d.in_cap) throw Error("Can't process data, buffer is too small");   // mfcccpu.cpp:338-339
        DeviceGuard g(h->device);
        int wc, wc_nd;
        h->spec_valid = false; h->out_is_spec = false; h->spec_on_host = false;
        h->pending = true;
        const int16_t *pcm = h->seg.set_input(data, samples, wc, wc_nd, h->st);
        h->blk_pcm = pcm; // stays intact in its ping-pong buffer until the set_input after the next one
        if (!h->fused() && wc > 0) launch_fft_mag(h->d, h->fft, h->mel, pcm, h->mag.p, wc_nd, h->st, h->pre); // segment + fft fused
        h->seg.carry(h->st);
        *frames = wc > 0 ? wc : 0;
    });
}

int afe_mfcc_flush(afe_mfcc *h, int *frames)
{
    *frames = 0;
    return guarded([&] {
        if (h->last_block) return;                             // nothing to flush (mfcccpu.cpp:350-351)
        h->last_block = true;
        DeviceGuard g(h->device);
        int wc, wc_nd;
        const int16_t *pcm = h->seg.flush(wc, wc_nd);
        h->blk_pcm = pcm;
        if (wc <= 0) return;
        if (!h->fused()) launch_fft_mag(h->d, h->fft, h->mel, pcm, h->mag.p, wc_nd, h->st, h->pre);
        *frames = wc;
    });
}

// do_delta (mfcccpu.cpp:234-263)
static void dynamics(afe_mfcc *h, int wc, bool first, bool last)
{
    const Derived &d = h->d;
    if (d.p.dyn == AFE_DYN_NONE || (first && last)) return;
    const int D = d.D;
    const float *src = h->statics();
    if (first) launch_pad_rows(src, h->dpad.p, wc + D, d.cols, D, 0, h->st);
    else if (last) launch_pad_rows(src, h->dpad.p, wc + D, d.cols, 0, D, h->st);
    else launch_pad_rows(src, h->dpad.p, wc + 2 * D, d.cols, 0, 0, h->st);
    launch_delta(h->dpad.p, h->d1.p, wc + 2 * d.l2, d.cols, d.l1, h->st);
    if (d.p.dyn == AFE_DYN_ACC) launch_delta(h->d1.p, h->d2.p, wc, d.cols, d.l2, h->st);
}

// MfccCpu::normalize (mfcccpu.cpp:265-282)
static void normalise(afe_mfcc *h, int wc, bool use_last)
{
    const Derived &d = h->d;
    if (d.p.norm == AFE_NORM_NONE) return;
    float *src = h->statics();
    if (d.p.norm_after_dyn) {
        h->n0.normalize(src + h->static_row_offset() * d.cols, wc, use_last, h->st);
        if (d.p.dyn != AFE_DYN_NONE) h->n1.normalize(h->d1.p + d.l2 * d.cols, wc, use_last, h->st);
        if (d.p.dyn == AFE_DYN_ACC) h->n2.normalize(h->d2.p, wc, use_last, h->st);
    } else
        h->n0.normalize(src, wc, use_last, h->st);
}

// One block through K1. The block's device PCM holds wc_nd frames; its output rows are the frames [t_first, t_first + wc):
//   first block   t_first = 0, left edge replicated by index clamping, D look-ahead frames on the right
//   middle block  t_first = D, context on both sides comes from the carried-over samples
//   flush block   t_first = D, right edge replicated; normalised with the previous block's statistics
// (mfcccpu.cpp:371-425; do_delta :234-263). Rows land in outb[0 .. wc). The tiles are described in the kernel arguments
// (FusedArgs::blk_*), so an apply() is ONE driver call: the launch.
static void apply_fused(afe_mfcc *h, int wc, int wc_nd, bool first, bool last)
{
    const Derived &d = h->d;
    FusedEngine &eng = *h->eng;
    eng.ensure_mel(h->alpha);
    const int t_first = first ? 0 : d.D;
    // small tiles: ONE block should occupy the whole GPU (a 512-frame tile is ~90 us of serial work for one CTA)
    int ntiles, nout;
    eng.plan_uniform(wc_nd, t_first, wc, eng.latency_tile(wc), ntiles, nout);
    if ((size_t)ntiles + 1 > h->tiles_cap) throw Error("block needs more tiles than the object was sized for");
    // quirk Q1: flushing after a single set_input reads every static D rows early (static_row_offset() == 0 there)
    const bool q1_flush = h->seg.last_calc_flushed && !h->fix_q1;
    FusedArgs a = eng.base_args((last && q1_flush) ? 2 : 0, h->blk_pcm, true);
    a.out = h->outb.p;
    a.blk_ntiles = ntiles; a.blk_T = wc_nd; a.blk_t_first = t_first; a.blk_n_out = wc; a.blk_nout = nout;
    // the rows a flush() right after this block would return ride along as one more tile (rows [wc, wc + D) of outb)
    const bool spec = !last && d.D > 0 && wc_nd >= 2 * d.D;
    a.blk_spec = spec ? 1 : 0; a.blk_spec_q1 = q1_flush ? 1 : 0;
    const int total = ntiles + (spec ? 1 : 0);
    const bool norm = d.p.norm != AFE_NORM_NONE;
    if (norm) { a.g_mean = h->norm.mean.p; a.g_scale = h->norm.scale.p; a.use_last = last ? 1 : 0; } // mfcccpu.cpp:389
    if (!norm || last) eng.launch_plain(a, total, h->st);
    else {
        eng.set_stats(a, h->norm, 3, wc);                     // this block's output rows (normalizercpu.cpp:22-30)
        if (!spec && eng.default_regression() && total <= 4 && eng.cluster_schedulable(total, a, h->st))
            eng.launch_clustered(a, total, total, h->norm, h->st);
        else if (!spec && total <= 8) eng.launch_ticket(a, total, h->norm, h->st);
        else eng.launch_roles(a, total, h->norm, h->st);
    }
    h->launches++;
    h->pending = true;
    h->out_is_spec = false; h->spec_on_host = false;
    h->spec_valid = spec;
    if (spec) { h->spec_alpha = h->alpha; h->spec_fix_q1 = h->fix_q1; h->spec_row0 = wc; }
}

int afe_mfcc_apply(afe_mfcc *h)
{
    return guarded([&] {
        const Derived &d = h->d;
        DeviceGuard g(h->device);
        int wc_nd, wc;
        bool first = false, last = false, use_last = false;
        if (h->last_block) {                                   // mfcccpu.cpp:373-390
            wc_nd = h->seg.est(h->seg.remaining); wc = wc_nd - d.D; last = true; use_last = true;
            if (wc <= 0) return;
            if (h->fused() && h->spec_valid && wc == d.D && h->spec_alpha == h->alpha && h->spec_fix_q1 == h->fix_q1) {
                h->out_is_spec = true;                         // these rows were computed with the previous block
                return;
            }
            h->spec_valid = false; h->out_is_spec = false;
        } else if (h->seg.last_calc_flushed) {                 // :391-407
            wc_nd = h->seg.est(h->seg.samples); wc = wc_nd - d.D; first = true;
            if (wc <= 0) throw Error("Can't process data, window count is too small");
        } else {                                               // :408-424
            wc_nd = h->seg.est(h->seg.samples); wc = wc_nd - 2 * d.D;
            if (wc <= 0) return;
        }
        if (h->fused()) { apply_fused(h, wc, wc_nd, first, last); return; }
        if (h->mel.alpha_built != h->alpha) upload_mel_tables(d, h->alpha, h->mel, h->st);  // refresh_filters per alpha
        launch_mel_dct(d, h->mel, h->mag.p, h->melv.p, h->cep.p, wc_nd, h->st);
        const bool norm = d.p.norm != AFE_NORM_NONE;
        if (!d.p.norm_after_dyn && norm) normalise(h, wc_nd, use_last);
        if (d.p.dyn != AFE_DYN_NONE) dynamics(h, wc, first, last);
        if (d.p.norm_after_dyn && norm) normalise(h, wc, use_last);
        // rows -> outb, so that get_output is one copy on either route
        const float *s0 = h->statics() + h->static_row_offset() * d.cols;
        const int ns = d.width / d.cols;
        launch_pack(s0, ns > 1 ? h->d1.p + d.l2 * d.cols : nullptr, ns > 2 ? h->d2.p : nullptr, h->outb.p, wc, d.cols, ns, h->st);
    });
}

int afe_mfcc_get_output(afe_mfcc *h, float *out, int frames)
{
    return guarded([&] {
        const Derived &d = h->d;
        if (frames > d.frame_cap) throw Error("Window count too high");   // mfcccpu.cpp:429-430
        if (frames <= 0) return;
        DeviceGuard g(h->device);
        const size_t n = (size_t)frames * d.width;
        if (h->out_is_spec) {                                  // flush rows computed (and usually already fetched) with the block
            if (frames > d.D) throw Error("Window count too high");
            const size_t off = (size_t)h->spec_row0 * d.width;
            if (!h->spec_on_host) {
                AFE_CUDA(cudaMemcpyAsync(h->h_out.p + off, h->outb.p + off, sizeof(float) * d.D * d.width, cudaMemcpyDeviceToHost, h->st));
                AFE_CUDA(cudaStreamSynchronize(h->st));
                h->pending = false; h->seg.synced(); h->spec_on_host = true;
            }
            memcpy(out, h->h_out.p + off, sizeof(float) * n);
            return;
        }
        // the speculative flush rows sit right behind the block's rows: one copy fetches both
        const bool with_spec = h->spec_valid && frames == h->spec_row0;
        const size_t n_copy = n + (with_spec ? (size_t)d.D * d.width : 0);
        AFE_CUDA(cudaMemcpyAsync(h->h_out.p, h->outb.p, sizeof(float) * n_copy, cudaMemcpyDeviceToHost, h->st));
        AFE_CUDA(cudaStreamSynchronize(h->st));
        h->pending = false; h->seg.synced(); h->spec_on_host = with_spec;
        memcpy(out, h->h_out.p, sizeof(float) * n);
    });
}

} // extern "C"

// ================================================================================================== stage objects
struct afe_segmenter {
    int device;
    Stream st;
    SegState seg;
    DevBuf<float> window;
    bool window_set = false;
};
struct afe_delta {
    int device, dim, window_limit, L;
    Stream st;
    DevBuf<float> out;
};

extern "C" {

int afe_segmenter_create(int W, int S, int window_limit, int deltasize, int cuda_device, afe_segmenter **out)
{
    *out = nullptr;
    return guarded([&] {
        if (afe_device_count() <= cuda_device) throw Error("no usable CUDA device (the product has no CPU fallback)");
        DeviceGuard g(cuda_device);
        std::unique_ptr<afe_segmenter> s(new afe_segmenter());
        s->device = cuda_device;
        s->st.create();
        s->seg.init(W, S, window_limit, deltasize);
        s->window.alloc(W);
        *out = s.release();
    });
}
void afe_segmenter_destroy(afe_segmenter *s)
{
    if (!s) return;
    cudaSetDevice(s->device);
    cudaStreamSynchronize(s->st);
    delete s;
}
int afe_segmenter_set_window(afe_segmenter *s, const float *w)
{
    return guarded([&] {
        DeviceGuard g(s->device);
        AFE_CUDA(cudaMemcpy(s->window.p, w, sizeof(float) * s->seg.W, cudaMemcpyHostToDevice));
        s->window_set = true;
    });
}
int afe_segmenter_set_input(afe_segmenter *s, const int16_t *in, float *d_out, int samples, int *wc, int *wc_nd)
{
    return guarded([&] {
        if (!s->window_set) throw Error("set_window must be called before set_input");
        DeviceGuard g(s->device);
        const int16_t *pcm = s->seg.set_input(in, samples, *wc, *wc_nd, s->st);
        if (*wc > 0) launch_segment(pcm, s->window.p, d_out, *wc_nd, s->seg.W, s->seg.S, s->seg.N2, s->st, s->seg.pre);
        s->seg.carry(s->st);
        AFE_CUDA(cudaStreamSynchronize(s->st));
        s->seg.synced();
    });
}
int afe_segmenter_flush(afe_segmenter *s, float *d_out, int *wc, int *wc_nd)
{
    return guarded([&] {
        DeviceGuard g(s->device);
        const int16_t *pcm = s->seg.flush(*wc, *wc_nd);
        if (*wc > 0) launch_segment(pcm, s->window.p, d_out, *wc_nd, s->seg.W, s->seg.S, s->seg.N2, s->st, s->seg.pre);
        AFE_CUDA(cudaStreamSynchronize(s->st));
    });
}
int afe_segmenter_set_preemphasis(afe_segmenter *s, float coefficient)
{
    return guarded([&] {
        if (!(coefficient >= 0.f && coefficient < 1.f)) throw Error("pre-emphasis coefficient must be in [0, 1)");
        s->seg.pre = coefficient;
    });
}
int afe_segmenter_remaining_samples(const afe_segmenter *s) { return s->seg.remaining; }
int afe_segmenter_samples(const afe_segmenter *s) { return s->seg.samples; }
int afe_segmenter_is_flushed(const afe_segmenter *s) { return s->seg.flushed; }
int afe_segmenter_was_flushed(const afe_segmenter *s) { return s->seg.last_calc_flushed; }

int afe_delta_create(int dim, int window_limit, int delta_size, int cuda_device, afe_delta **out)
{
    *out = nullptr;
    return guarded([&] {
        if (afe_device_count() <= cuda_device) throw Error("no usable CUDA device (the product has no CPU fallback)");
        DeviceGuard g(cuda_device);
        std::unique_ptr<afe_delta> d(new afe_delta());
        d->device = cuda_device; d->dim = dim; d->window_limit = window_limit; d->L = delta_size;
        d->st.create();
        d->out.alloc((size_t)dim * window_limit);
        *out = d.release();
    });
}
void afe_delta_destroy(afe_delta *d)
{
    if (!d) return;
    cudaSetDevice(d->device);
    cudaStreamSynchronize(d->st);
    delete d;
}
int afe_delta_apply(afe_delta *d, const float *d_data, int window_count)
{
    return guarded([&] {
        if (window_count > d->window_limit) throw Error("Window count too high");
        DeviceGuard g(d->device);
        launch_delta(d_data, d->out.p, window_count, d->dim, d->L, d->st);
        AFE_CUDA(cudaStreamSynchronize(d->st));
    });
}
float *afe_delta_output(afe_delta *d) { return d->out.p; }

int afe_normalizer_create(int norm_type, int dim, int cuda_device, afe_normalizer **out)
{
    *out = nullptr;
    return guarded([&] {
        if (afe_device_count() <= cuda_device) throw Error("no usable CUDA device (the product has no CPU fallback)");
        if (norm_type < AFE_NORM_NONE || norm_type > AFE_NORM_MINMAX || dim < 1) throw Error("invalid normalizer arguments");
        DeviceGuard g(cuda_device);
        std::unique_ptr<afe_normalizer> n(new afe_normalizer());
        n->device = cuda_device;
        n->own_st.create();
        n->st = n->own_st;
        n->ns.init(norm_type, dim);
        n->ns.reset_record(n->st);
        *out = n.release();
    });
}
void afe_normalizer_destroy(afe_normalizer *n)
{
    if (!n) return;
    cudaSetDevice(n->device);
    cudaStreamSynchronize(n->own_st);
    delete n;
}
static cudaStream_t norm_stream(afe_normalizer *n) { return n->st ? n->st : n->own_st; }

int afe_normalizer_normalize(afe_normalizer *n, float *d_data, int offset, int window_count, int use_last_stats)
{
    return guarded([&] {
        DeviceGuard g(n->device);
        n->ns.normalize(d_data + offset, window_count, use_last_stats != 0, norm_stream(n));
        AFE_CUDA(cudaStreamSynchronize(norm_stream(n)));
    });
}

// ---- corpus-level statistics: the verbs of the OpenCL class' three kernels (norm.cl kernelSum / kernelFinalizeSum /
// kernelNormalize, normalizeropencl.cpp:123-158) exposed one by one, with the all-reduce between the first two.
int afe_normalizer_stats_len(const afe_normalizer *n) { return n->ns.rec_len(); }
int afe_normalizer_reset(afe_normalizer *n)
{
    return guarded([&] { DeviceGuard g(n->device); n->ns.reset_record(norm_stream(n)); });
}
int afe_normalizer_accumulate(afe_normalizer *n, const float *d_data, int offset, int window_count)
{
    return guarded([&] {
        if (window_count < 0) throw Error("accumulate: negative window count");
        DeviceGuard g(n->device);
        n->ns.accumulate(d_data + offset, window_count, norm_stream(n));
    });
}
int afe_normalizer_allreduce(afe_normalizer *n, void *nccl_comm)
{
    return guarded([&] {
        DeviceGuard g(n->device);
        const int w = n->ns.dim;
        double *rec = n->ns.rec.p;
        // one NCCL group: sums + count (ncclSum), minima (ncclMin), maxima (ncclMax) — 4*dim+1 doubles, latency bound
        nccl_allreduce_stats(nccl_comm, rec, 2 * w + 1, rec + 2 * w + 1, w, rec + 3 * w + 1, w, norm_stream(n));
    });
}
int afe_normalizer_finalize(afe_normalizer *n)
{
    return guarded([&] { DeviceGuard g(n->device); n->ns.finalize(norm_stream(n)); });
}
int afe_normalizer_apply(afe_normalizer *n, float *d_data, int offset, int window_count)
{
    return guarded([&] {
        DeviceGuard g(n->device);
        n->ns.apply(d_data + offset, window_count, norm_stream(n));
        AFE_CUDA(cudaStreamSynchronize(norm_stream(n)));
    });
}
int afe_normalizer_get_stats(afe_normalizer *n, double *h_stats)
{
    return guarded([&] {
        DeviceGuard g(n->device);
        AFE_CUDA(cudaMemcpyAsync(h_stats, n->ns.rec.p, sizeof(double) * n->ns.rec_len(), cudaMemcpyDeviceToHost, norm_stream(n)));
        AFE_CUDA(cudaStreamSynchronize(norm_stream(n)));
    });
}
int afe_normalizer_set_stats(afe_normalizer *n, const double *h_stats)
{
    return guarded([&] {
        DeviceGuard g(n->device);
        AFE_CUDA(cudaMemcpyAsync(n->ns.rec.p, h_stats, sizeof(double) * n->ns.rec_len(), cudaMemcpyHostToDevice, norm_stream(n)));
        AFE_CUDA(cudaStreamSynchronize(norm_stream(n)));
    });
}

int afe_device_malloc(int dev, size_t bytes, void **p)
{
    return guarded([&] { DeviceGuard g(dev); AFE_CUDA(cudaMalloc(p, bytes ? bytes : 1)); });
}
int afe_device_free(int dev, void *p)
{
    return guarded([&] { DeviceGuard g(dev); AFE_CUDA(cudaFree(p)); });
}
int afe_memcpy_h2d(int dev, void *d, const void *h, size_t bytes)
{
    return guarded([&] { DeviceGuard g(dev); AFE_CUDA(cudaMemcpy(d, h, bytes, cudaMemcpyHostToDevice)); });
}
int afe_memcpy_d2h(int dev, void *h, const void *d, size_t bytes)
{
    return guarded([&] { DeviceGuard g(dev); AFE_CUDA(cudaMemcpy(h, d, bytes, cudaMemcpyDeviceToHost)); });
}

} // extern "C"
