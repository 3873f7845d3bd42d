/* cproc_cuda.h -- C-ABI of the B200 batched renderer for the synth_tools
 * per-sample DSP hot path.  Plain C99 (includable from the linux/ C hosts built with
 * -std=gnu99, rules.mk:304); no CUDA or C++ types cross this boundary.
 *
 * The library renders N independent instances of one reference processor for
 * F frames per call ("N instances x F frames").  Every processor keeps the
 * reference's state / param / input / output record layouts, so a host that
 * owns reference structs uploads them as they are (base pointer + stride).
 *
 *   reference interface                         entry point that replaces it
 *   ------------------------------------------  -----------------------------
 *   NAME_update(state*,config*,param*,input*)   cproc_cuda_alloc + _run
 *     generic/cproc.h:89-95
 *   void cproc_update(w *input, w changed)      CPROC_CUDA_GRAPH batch
 *     linux/test_cproc.c:13-17,
 *     stm32f103/mod_cproc_plugin.c:20-38
 *   uint32_t pdmK_update(struct pdmK*, in,      CPROC_CUDA_PDM batch
 *     out_shift[, dither]) stm32f103/pdm.h:13-77
 *   pdm_channels_update / channel_update_dither CPROC_CUDA_PDM_V1 batch
 *     stm32f103/mod_pdm.c:230-264
 *   HW_TIM_ISR(TIM_PDM) + control_update        CPROC_CUDA_PDM_V2 batch
 *     stm32f103/mod_pdm_pwm.c:123-143,
 *     stm32f103/mod_controlrate.c:28-57
 *   pwm_update  stm32f103/mod_pdm.c:167-175     CPROC_CUDA_PWM batch
 *   word clock  linux/clock.c:109-120           CPROC_CUDA_WORD_CLOCK batch
 *   synth_run / sum_tick_saw / sum_tick_square  CPROC_CUDA_VOICE_BANK batch
 *     linux/synth.c:169-202
 *   square_grain_proc linux/synth_tools.c:85-100 CPROC_CUDA_SQUARE_GRAIN batch
 *
 * The reference hot path is `void` and cannot fail; its surroundings return
 * int 0 / negative (stm32f103/mod_synth.c:89-137).  Every function here
 * returns 0 or a negative CPROC_CUDA_E* code and never aborts.  There is no
 * CPU fallback: without a CUDA device cproc_cuda_open fails with
 * CPROC_CUDA_ENODEV.
 *
 * Threading: like the reference (one JACK RT thread / one ISR per graph), a
 * context and its batches have a single caller at a time.
 *
 * ABI version 2: cproc_cuda_node carries a second source (two-input processors),
 * cproc_cuda_config an output-node list; graph front end, patcher and mix bus added.
 * ABI version 3: float processors as graph nodes (phasor_f, svf, env, onepole, gain,
 * asfloat; include/cproc_ext.h), graph batches carry a param record, cproc_cuda_graph_info
 * grows (param words and initialisers, output types), evented graph driver.
 */
#ifndef CPROC_CUDA_H
#define CPROC_CUDA_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CPROC_CUDA_ABI_VERSION 3

/* ---- error codes -------------------------------------------------------- */
#define CPROC_CUDA_OK        0
#define CPROC_CUDA_EINVAL   (-1)  /* bad argument / unsupported combination   */
#define CPROC_CUDA_ENODEV   (-2)  /* no usable CUDA device                    */
#define CPROC_CUDA_ENOMEM   (-3)  /* device or pinned-host allocation failed  */
#define CPROC_CUDA_ECUDA    (-4)  /* CUDA runtime error (see _last_error)     */
#define CPROC_CUDA_ESTATE   (-5)  /* call order violated (e.g. run w/o state) */

typedef struct cproc_cuda_ctx   cproc_cuda_ctx;    /* one device + stream   */
typedef struct cproc_cuda_batch cproc_cuda_batch;  /* N instances of a proc */

/* ---- processors --------------------------------------------------------- */
enum cproc_cuda_proc {
    /* Generated cproc graph of acc/edge nodes == cproc_update(w *input, w
     * changed).  state record: node states concatenated in ANF order
     * (acc_state {w out}, edge_state {w out; w last}; cproc.h:134,145; glide: 5 words;
     * pdm: K+1 words).
     * in:  uint32 [inst][n_inputs][F]; in2: changed mask uint32 [inst][F] or
     * NULL (= -1, mod_cproc_plugin.c:32); out: uint32 [inst][F], the value
     * passed to cproc_output() each tick (test_cproc.c:16); with several
     * cproc_output statements [inst][n_outputs][F].  A graph that reads no
     * input[] (a free-running phasor_f voice) has n_inputs == 0 and in == NULL.
     * param record: the nodes' param structs concatenated in ANF order (only the
     * extension processors have one, see the node kinds below).
     * mix (or NULL): the bus mix of every output, 32-bit words [bus][n_outputs][F], bus = instance /
     * cfg.voices_per_bus (0: every instance on one bus); out may then be NULL (no per-instance stream is
     * written), and with both set out holds what an out-only run writes.  Output q is a float when its
     * node kind outputs a float (whichever of cproc_output / cproc_output_f named it): summed in binary32,
     * one __fadd_rn rounding per add, no flush to zero; a w output is summed mod 2^32.  Summation order
     * (part of the contract, so results are bit-reproducible): a balanced pairwise tree over the bus's
     * instances in index order -- the instance count padded to a power of two with -0.0f (0 for w; adding
     * -0 is an exact identity, so a one-instance bus gives its output), level 1 adds instances (2m, 2m+1),
     * level 2 those pair sums, and so on.  The tree depends on the bus's instance count only: not on F,
     * on how frames are split over calls, on the layout or on any cproc_cuda_set_option value.  With n
     * instances on one bus, |mix - exact sum| <= gamma_d * sum |out|, d = ceil(log2 n), gamma_d = d u /
     * (1 - d u), u = 2^-24.  A multi-GPU host all-reduces the mix with cproc_cuda_bus_allreduce, op 2 when
     * every output is a float, op 0 when every output is a w.  The run call returns CPROC_CUDA_EINVAL with
     * mix set for voices_per_bus neither 0 nor a multiple of 32, for cfg.mode = CPROC_CUDA_GRAPH_SCAN and
     * for the TILED layout; there is no mix in cproc_cuda_run_stream or cproc_cuda_patch_tick, and
     * cproc_cuda_bus_attach does not take GRAPH batches. */
    CPROC_CUDA_GRAPH = 1,
    /* pdmK_update, K = cfg.order (pdm.h).  state record: struct pdmK.
     * param record: {uint32 input} used when in == NULL.  in: uint32
     * [inst][F] or NULL; in2: dither uint32 [F] shared by all instances or
     * NULL (0); out: uint32 [inst][F] quantiser output. */
    CPROC_CUDA_PDM = 2,
    /* mod_pdm.c v1 carry-bit PDM.  state record: struct channel {uint32
     * setpoint; uint32 accu} (mod_pdm.c:198-201).  Banks of cfg.bank_size
     * channels share one dither word per tick (mod_pdm.c:261):
     * dither = (in2 ? in2[bank][t] : xorshift32(&prng[bank])) & dither_mask.
     * out: packed bits, uint32 words, sample t at bit (t & 31) of word t>>5:
     * PLANAR [ch][F/32], INTERLEAVED [F/32][ch].  F % 32 == 0. */
    CPROC_CUDA_PDM_V1 = 3,
    /* mod_pdm_pwm.c v2 (glide + pdmK + control-rate line).  state record:
     * struct channel {uint32 setpoint; struct line {uint32 position; int32
     * velocity} line[2]; struct pdmK pdm} (mod_pdm_pwm.c:80-93) = 5+K words.
     * ctl: setpoints uint32 [n_ctl][ch] (one row latched at every control
     * boundary met during the run, before the line copy) or NULL.
     * in2: external dither uint32 [bank][F] or NULL (xorshift32 per bank).
     * out: uint8 duty.  PLANAR [ch][F], TILED [F/16][ch][16], INTERLEAVED
     * [F][ch] (the order the ISR emits: one byte per channel per tick). */
    CPROC_CUDA_PDM_V2 = 4,
    /* pwm_update (mod_pdm.c:167-175).  state {uint32 phase}; param {uint32
     * speed}; out uint8 duty: PLANAR [inst][F], INTERLEAVED [F][inst], TILED
     * [F/16][inst][16]. */
    CPROC_CUDA_PWM = 5,
    /* linux/synth.c voice bank.  state record: struct voice {uint32 note_inc;
     * uint32 note_state} (synth.c:33-36).  Consecutive groups of
     * cfg.voices_per_bus voices feed one bus (reference: 64, synth.c:39).
     * cfg.mode: CPROC_CUDA_MIX_SAW (sum_tick_saw) / _SQUARE.
     * out: float [bus][F] (what synth_run writes to vec); mix: int32
     * [bus][F] raw integer mix before the float scale (synth.c:171,184) --
     * the buffer a multi-GPU host all-reduces.  Either may be NULL. */
    CPROC_CUDA_VOICE_BANK = 6,
    /* square_grain_proc (synth_tools.c:85-100).  state {float state}; param
     * {float threshold}; in/out float [inst][F]; in may alias out. */
    CPROC_CUDA_SQUARE_GRAIN = 7,
    /* square_grain fed by a per-grain phasor (acc -> signed saw) and mixed
     * to stereo with dyadic pan gains k/64, integer mix in units of 2^-7.
     * state {float state; uint32 phase}; param {float threshold; uint32 inc;
     * uint32 gl; uint32 gr}; out float [2][F]; mix int32 [2][F].  Either
     * may be NULL, not both.  With a mix bus attached (cproc_cuda_bus_attach)
     * they receive the bus of ALL ranks: mix the summed int32 words, out
     * (float)word * 2^-7.
     * gl, gr <= 64: upload_param returns CPROC_CUDA_EINVAL above 64.
     * Every float state acts and comes back as in the reference (a NaN state never flips
     * and adds 0); a state other than +-0, +-0.5 selects a slower kernel until the next upload. */
    CPROC_CUDA_SQUARE_GRAIN_MIX = 8,
    /* Extension voice (not in the reference): phasor -> Chamberlin SVF ->
     * linear AR envelope -> pan.  state {uint32 phase; float lp, bp, env;
     * uint32 t}; param {uint32 inc; float f, q, env_attack, env_release;
     * uint32 gate_frames; float gl, gr}.  out: raw float [inst][F][2]
     * (PLANAR) / [F/2][inst][2][2] (TILED) or NULL; mix: float [2][F] or NULL.
     * cfg.mode = CPROC_CUDA_XVOICE_SCAN renders raw output time-parallel (few
     * voices, long streams): chunk start states from a block scan of the SVF's
     * affine recurrence in fp64; phase/t/env stay bit-exact; lp/bp and the output of
     * every voice are within 1e-5 of that voice's own peak of the exact (fp64) filter,
     * or within twice the sequential render's own error where that is larger (measured
     * on a B200: <= 1.3e-6 of the voice's peak for 1e-3 <= f <= 0.9, 5e-3 <= q <= 2,
     * up to 2^18 frames; the sequential render <= 6.2e-6 there). */
    CPROC_CUDA_XVOICE = 9,
    /* one-pole low-pass y += a*(x-y) (extension).  state {float y}; param
     * {float a}; in/out float [inst][F].  cfg.mode = CPROC_CUDA_ONEPOLE_SCAN: few
     * instances, long streams -- time-parallel render from a block scan of the affine
     * recurrence (fp64 chunk start states; in must not alias out).  Every instance is within
     * 1e-5 of its own peak of the exact (fp64) recurrence, or within twice the sequential
     * render's own error where that is larger (measured on a B200: <= 4.7e-6 for 2^-24 <= a
     * <= 1.999).  The sequential float render itself stalls wherever |a (x - y)| < 1/2 ulp(y)
     * -- a smoother with a small coefficient -- and then drifts from the exact result: up to
     * 3.5e-4 of the peak at a = 1e-6, 1.8e-3 at a = 2^-24 over 40,000 frames, 3e-5 for a step
     * at a = 1e-3; the scan does not, as it restarts every chunk from an fp64 state. */
    CPROC_CUDA_ONEPOLE = 10,
    /* word clock of linux/clock.c:109-120 (integer divisor of the sample clock): per sample
     * `if (phase >= hperiod) { phase -= hperiod; pol ^= 1; } out = pol; phase += 1`.
     * state {int32 phase; int32 pol}; param {int32 hperiod} (clock.c:58: sr*5 / (bpm*4));
     * out float PLANAR [inst][F] / INTERLEAVED [F][inst].  The MIDI clock byte of clock.c:113-116
     * goes out where pol turns 1: the host adapter reads those samples off its block. */
    CPROC_CUDA_WORD_CLOCK = 11
};

/* Node kinds (bits 0..7 of cproc_cuda_node.type; bits 8..15 carry the node's config word).
 * GLIDE is the firmware's control-rate -> audio-rate parameter interpolation
 * (struct line[2] of mod_pdm_pwm.c:80-93, pdm_update_line of mod_controlrate.c:28-40,
 * the "representative example" of doc/combinators.org:28-34) as a processor: .in is
 * read once per 2^L ticks, .out is the interpolated line; state record {out, vel0,
 * pos1, vel1, count}; L = CPROC_CUDA_NODE_ARG(type) = CONTROL_DIV_LOG.
 * PDM is pdmK_update (stm32f103/pdm.h:13-77) as a processor: .in the modulator input,
 * .dither the second input (src2), .out the quantiser output; state record {out, s1..sK};
 * config word = K | out_shift << 3.  glide -> pdm2 is the firmware's whole v2 channel
 * (mod_pdm_pwm.c:97-116) as a graph.
 *
 * Extension processors (SURVEY 8 a-X; not in the reference): the DEF_PROC definitions are
 * include/cproc_ext.h, written against the reference's generic/cproc.h:89-103 so that the same
 * graph text compiles as C on a CPU host.  Their `float` fields are IEEE binary32 carried in the
 * same 32-bit words as `w` (state rows, param rows and output streams hold the bit patterns);
 * every float operation is one rounding in a fixed order (fmaf where cproc_ext.h says fmaf), so
 * results are bit-identical to the C definitions compiled with -ffp-contract=off (for non-NaN data: a NaN
 * result is the canonical 0x7FFFFFFF on the GPU where an x86 host propagates the operand's payload).
 *   phasor_f  state {float out; w phase}          param {w inc}   input {w mod}
 *             out = (float)(int32_t)phase * 2^-31; phase += inc + mod    (signed saw, read before advance)
 *   svf       state {float out; float bp}         param {float f; float q}   input {float in}
 *             Chamberlin: lp = fmaf(f, bp, out); hp = in - lp; hp = fmaf(-q, bp, hp); bp = fmaf(f, hp, bp); out = lp
 *   env       state {float out; float env; w t}   param {float attack; float release; w gate_frames}   input {float in}
 *             linear attack / release: t < gate_frames ? env = min(env + attack, 1) : env = max(env - release, 0); t += 1; out = in * env
 *   onepole   state {float out}                   param {float a}   input {float in}     out = fmaf(a, in - out, out)
 *   gain      state {float out}                   param {float g}   input {float in}     out = g * in
 *   asfloat   state {float out}                   input {w in}      out = the float whose bits are `in` (external float streams)
 *   glide_f   state {float out; float step; w count}   config {w div_log}   input {float in}
 *             control rate -> audio rate: every 2^div_log ticks step = (in - out) * 2^-div_log; every tick out += step
 *   mul       state {float out}                   input {float in; float gain}      out = in * gain
 *             glide_f -> mul is the "representative example" of doc/combinators.org:28-34 (a control-rate gain amount applied
 *             to an audio-rate signal) for float signals, as glide is for the firmware's uint32 setpoints
 * Connecting a `w` output (or input[k]) to a float input converts by value, (float)(uint32_t)x, as the
 * C assignment in PROC_COND's designated initialiser does (cproc.h:75); a float output feeding a `w`
 * input is rejected (undefined in C for negative values).  An input the statement does not name reads
 * 0, like the omitted member of the C initialiser: src = CPROC_CUDA_SRC_ZERO.
 * The param record of a graph batch is the concatenation of its nodes' param structs in ANF order
 * (cproc_cuda_upload_param; cproc_cuda_param_bytes). */
enum { CPROC_CUDA_NODE_ACC = 0, CPROC_CUDA_NODE_EDGE = 1, CPROC_CUDA_NODE_GLIDE = 2, CPROC_CUDA_NODE_PDM = 3,
       CPROC_CUDA_NODE_PHASOR_F = 4, CPROC_CUDA_NODE_SVF = 5, CPROC_CUDA_NODE_ENV = 6, CPROC_CUDA_NODE_ONEPOLE = 7,
       CPROC_CUDA_NODE_GAIN = 8, CPROC_CUDA_NODE_ASFLOAT = 9, CPROC_CUDA_NODE_GLIDE_F = 10, CPROC_CUDA_NODE_MUL = 11,
       CPROC_CUDA_NODE_KINDS = 12 };
#define CPROC_CUDA_NODE_GLIDE_F_L(L) (CPROC_CUDA_NODE_GLIDE_F | ((uint32_t)(L) << 8))
#define CPROC_CUDA_SRC_ZERO ((int32_t)0x80000000)
#define CPROC_CUDA_NODE_KIND(t) ((t) & 0xFFu)
#define CPROC_CUDA_NODE_ARG(t)  (((t) >> 8) & 0xFFu)
#define CPROC_CUDA_NODE_GLIDE_L(L) (CPROC_CUDA_NODE_GLIDE | ((uint32_t)(L) << 8))
#define CPROC_CUDA_NODE_PDM_K(K, SH) (CPROC_CUDA_NODE_PDM | (((uint32_t)(K) | ((uint32_t)(SH) << 3)) << 8))
#define CPROC_CUDA_GRAPH_MAX_NODES 64
enum { CPROC_CUDA_MIX_SAW = 0, CPROC_CUDA_MIX_SQUARE = 1 };
enum { CPROC_CUDA_XVOICE_SEQ = 0, CPROC_CUDA_XVOICE_SCAN = 1 };
enum { CPROC_CUDA_ONEPOLE_SEQ = 0, CPROC_CUDA_ONEPOLE_SCAN = 1 };
/* GRAPH batches of acc / edge nodes only: cfg.mode = CPROC_CUDA_GRAPH_SCAN renders time-parallel
 * and still bit-exact (prefix sums and an associative composition of the edge detector's maps
 * over time chunks) -- for few instances and long streams, e.g. the reference's single voice. */
enum { CPROC_CUDA_GRAPH_SEQ = 0, CPROC_CUDA_GRAPH_SCAN = 1 };

/* Stream layouts (per-instance streams `x[inst][frame]`). */
enum {
    CPROC_CUDA_PLANAR = 0,      /* [inst][F]: what the reference hosts hand over
                                   (float *vec, t_float *in/out)              */
    CPROC_CUDA_INTERLEAVED = 1, /* [F][inst]: voice-interleaved frames        */
    CPROC_CUDA_TILED = 2        /* [F/T][inst][T], T*elem = 16 bytes: native,
                                   one 128-bit store per thread               */
};

/* One PROC_COND statement of a generated graph (cproc.h:72-77). */
typedef struct {
    uint32_t type;       /* CPROC_CUDA_NODE_* | config word << 8             */
    int32_t  src;        /* >=0: .in = n<src>.out; <0: .in = input[-(src+1)] */
    uint32_t cond_mask;  /* node runs iff (changed & cond_mask) != 0         */
    int32_t  src2;       /* second input (pdm: .dither), same encoding; ignored by one-input processors */
} cproc_cuda_node;

typedef struct {
    uint32_t proc;            /* enum cproc_cuda_proc                        */
    uint32_t layout;          /* default stream layout for in/out            */
    /* PDM family */
    uint32_t order;           /* 1..4  (PDM_ORDER, mod_pdm_pwm.c:85)         */
    uint32_t out_shift;       /* 32 - PDM_DIV_LOG = 24 (mod_pdm_pwm.c:115)   */
    uint32_t bank_size;       /* channels sharing one dither word per tick   */
    uint32_t dither_mask;     /* 0x3FF (mod_pdm_pwm.c:127) / 0x0FFFFFFF (mod_pdm.c:261) */
    uint32_t ctl_div_log;     /* CONTROL_DIV_LOG = 12 (mod_pdm_pwm.c:76)     */
    /* voice bank */
    uint32_t mode;            /* CPROC_CUDA_MIX_* / CPROC_CUDA_XVOICE_*      */
    uint64_t voices_per_bus;  /* 0 = all instances on one bus (voice bank, graph mix) */
    /* graph */
    const cproc_cuda_node *nodes;
    uint32_t n_nodes, n_inputs, out_node;
    uint32_t n_outputs;       /* 0 / 1: one output stream, the .out of node out_node          */
    const uint32_t *out_nodes;/* n_outputs > 1: the nodes behind the cproc_output() calls, in
                                 order; out is then uint32 [inst][n_outputs][F] (PLANAR) /
                                 [F][n_outputs][inst] (INTERLEAVED), like the input streams   */
} cproc_cuda_config;
#define CPROC_CUDA_GRAPH_MAX_OUTPUTS 16

/* Front end for the generated graph text (SURVEY 8 f-1).  `text` is what
 * epid_cproc.erl emits and the reference compiles as C (linux/test_cproc.c:11-17,
 * stm32f103/bp5_plugin.c:1-9): `#define CPROC_NB_INPUTS n`, a sequence of
 *   PROC_COND(<changed> & <mask>, <inst>, acc|edge, NULL, NULL, .in = input[k] | <inst>.out);
 *   PROC_COND(<changed> & <mask>, <inst>, glide, &(glide_config){.div_log = L}, NULL, .in = ...);
 *   PROC_COND(<changed> & <mask>, <inst>, pdm1..pdm4, &(pdm_config){.out_shift = S}, NULL, .in = ..., .dither = ...);
 *   PROC(<inst>, glide_f, &(glide_f_config){.div_log = L}, NULL, .in = ...);   PROC(<inst>, mul, NULL, NULL, .in = ..., .gain = ...);
 *   PROC(<inst>, phasor_f|svf|env|onepole|gain|asfloat, NULL, <param>, .in = ... [, .mod = ...]);
 *     <param>: &<identifier> (the host uploads the record) or a compound literal whose members become the
 *     record's initial value for every instance, e.g. (&(svf_param){ .f = 0.1f, .q = 1.5f }) -- in parentheses, or
 *     the C preprocessor splits the macro argument at the literal's commas; NULL for asfloat
 * (or PROC(<inst>, ...), cproc.h:81) and one or more `cproc_output(<index>, <inst>.out);` -- for a float
 * node `cproc_output_f(<index>, <inst>.out);` (the stream then carries the float's bits).
 * Fills `nodes` (at most max_nodes rows) and `info`; the rows go into
 * cproc_cuda_config.nodes / n_nodes / n_inputs / out_node unchanged.  Needs no device. */
typedef struct {
    uint32_t n_nodes, n_inputs, out_node;
    uint32_t out_index;       /* first argument of cproc_output (the TAG_U32 index, mod_cproc_plugin.c:40-43) */
    uint32_t n_outputs;       /* number of cproc_output statements (out_node / out_index are the first)      */
    uint32_t out_nodes[16], out_indices[16];
    uint32_t out_is_float;    /* bit q: output q came from cproc_output_f                                    */
    uint32_t n_param_words;   /* words of the batch's param record                                           */
    uint32_t param_init[192]; /* the record's initial value: compound-literal members, 0 elsewhere           */
} cproc_cuda_graph_info;
#define CPROC_CUDA_GRAPH_MAX_PARAM_WORDS 192
int  cproc_cuda_graph_parse(const char *text, cproc_cuda_node *nodes, uint32_t max_nodes, cproc_cuda_graph_info *info);

/* Buffers of one run.  Host pointers for cproc_cuda_run, device pointers for
 * cproc_cuda_run_dev.  Unused members are NULL. */
typedef struct {
    const void *in;     /* per-instance input stream                        */
    const void *in2;    /* second input: changed mask / dither              */
    const void *ctl;    /* control-rate input rows (setpoints)              */
    void       *out;    /* per-instance (or per-bus) output stream          */
    void       *mix;    /* mix bus                                          */
    uint32_t    layout; /* CPROC_CUDA_* layout of in/out for this run       */
    uint32_t    n_ctl;  /* rows available in ctl                            */
} cproc_cuda_io;

/* ---- context ------------------------------------------------------------ */
/* stream: a cudaStream_t the caller owns (e.g. the host framework's current
 * stream) or NULL to let the context create its own. */
int  cproc_cuda_open(int device, void *stream, cproc_cuda_ctx **ctx);
int  cproc_cuda_close(cproc_cuda_ctx *ctx);
int  cproc_cuda_sync(cproc_cuda_ctx *ctx);
/* Last error text of this context (ctx may be NULL: process-wide last). */
const char *cproc_cuda_last_error(const cproc_cuda_ctx *ctx);
int  cproc_cuda_abi_version(void);
int  cproc_cuda_device_count(void);
/* Number of kernels this context has launched (bench accounting). */
uint64_t cproc_cuda_launch_count(const cproc_cuda_ctx *ctx);

/* ---- batches ------------------------------------------------------------ */
int  cproc_cuda_alloc(cproc_cuda_ctx *ctx, const cproc_cuda_config *cfg,
                      uint64_t n_instances, cproc_cuda_batch **batch);
int  cproc_cuda_free(cproc_cuda_batch *batch);
/* Bytes of one state / param record as laid out by the reference. */
size_t cproc_cuda_state_bytes(const cproc_cuda_batch *batch);
size_t cproc_cuda_param_bytes(const cproc_cuda_batch *batch);
/* Records are read/written at `aos + i*stride` (stride 0 = packed).  State
 * starts zeroed (cproc.h:65-66).  These are the checkpoint/resume calls. */
int  cproc_cuda_upload_state(cproc_cuda_batch *b, const void *aos, size_t stride);
int  cproc_cuda_download_state(cproc_cuda_batch *b, void *aos, size_t stride);
int  cproc_cuda_upload_param(cproc_cuda_batch *b, const void *aos, size_t stride);
/* Per-bank dither PRNG words (n_banks = ceil(N / bank_size)) and the shared
 * control divider counter (control_div_count, mod_pdm_pwm.c:78). */
int  cproc_cuda_upload_bank(cproc_cuda_batch *b, const uint32_t *prng, uint32_t count);
int  cproc_cuda_download_bank(cproc_cuda_batch *b, uint32_t *prng, uint32_t *count);

/* Render F frames.  _run: host buffers, synchronous (copies in, renders,
 * copies out, returns when `out` is valid) -- the drop-in path.
 * _run_dev: device buffers, asynchronous on the context stream. */
int  cproc_cuda_run(cproc_cuda_batch *b, uint64_t n_frames, const cproc_cuda_io *io);
int  cproc_cuda_run_dev(cproc_cuda_batch *b, uint64_t n_frames, const cproc_cuda_io *io);
/* One period of a real-time host that keeps the state in ITS structs -- synth_run(struct synth *x, ...) renders from
 * x->voice[] and leaves the phases there (linux/synth.c:196-202), note_on / note_off write the same structs between
 * periods (:143-165).  Equivalent to upload_state(state_aos, stride); run(n_frames, io); download_state(state_aos,
 * stride), but as one stream sequence with ONE synchronisation and, after the first call with a batch, no allocation
 * (pinned record staging owned by the batch): call it once before the real-time thread starts. */
int  cproc_cuda_run_period(cproc_cuda_batch *b, uint64_t n_frames, const cproc_cuda_io *io, void *state_aos, size_t stride);
/* Long renders into host memory: F_total frames in chunks of F_chunk, the
 * device->host copy of chunk k overlapped with the render of chunk k+1.
 * io->out is a PINNED host buffer (cproc_cuda_host_alloc) of `ring_chunks`
 * slabs, each one chunk in io->layout with F = F_chunk; chunk k lands in slab
 * k % ring_chunks.  ring_chunks == 0 means one slab per chunk (the whole
 * render is kept).  `on_chunk` (may be NULL) is called on the calling thread
 * once chunk k is in host memory -- the equivalent of the JACK process
 * callback handing over a period -- and must be done with the slab when it
 * returns.  ring_chunks must be 0 or >= 2.  Synchronous. */
typedef void (*cproc_cuda_chunk_fn)(void *user, uint64_t chunk_index, const void *slab, size_t slab_bytes);
int  cproc_cuda_run_stream(cproc_cuda_batch *b, uint64_t n_frames_total,
                           uint64_t n_frames_chunk, const cproc_cuda_io *io,
                           uint32_t ring_chunks, cproc_cuda_chunk_fn on_chunk, void *user);
/* Evented driver of a GRAPH batch == handle_tag_u32 of stm32f103/mod_cproc_plugin.c:24-38,
 *     cproc_input[i] = v; cproc_update(cproc_input, -1);
 * The batch keeps the reference's persistent `w cproc_input[CPROC_NB_INPUTS]` (:20) per instance,
 * zero when the batch is allocated.  _set_input writes input[i] of one instance, or of every
 * instance when instance == CPROC_CUDA_ALL_INSTANCES; i >= n_inputs returns CPROC_CUDA_EINVAL
 * where the reference returns -1 (:29,35-36).  _tick runs ONE tick of every instance on those
 * inputs under the `changed` mask (-1 in the reference, :32) and copies the values handed to
 * cproc_output() to out: uint32 [inst][n_outputs] (out may be NULL).  _event is the two in one
 * call for a single instance: what one TAG_U32 message [i, v] does; out: uint32 [n_outputs]. */
#define CPROC_CUDA_ALL_INSTANCES (~(uint64_t)0)
int  cproc_cuda_graph_set_input(cproc_cuda_batch *b, uint64_t instance, uint32_t i, uint32_t v);
int  cproc_cuda_graph_tick(cproc_cuda_batch *b, uint32_t changed, uint32_t *out);
int  cproc_cuda_graph_event(cproc_cuda_batch *b, uint64_t instance, uint32_t i, uint32_t v, uint32_t *out);
/* Graph batches are compiled for their node table with NVRTC when first run (one
 * kernel per graph: node states in registers, sources and masks as literals).  The
 * compiler log (warnings, or the reason the table-driven kernel is used instead) and
 * the generated CUDA source for a node table (returns its length; copies at most
 * cap-1 bytes; needs no device). */
const char *cproc_cuda_graph_jit_log(const cproc_cuda_batch *b);
int  cproc_cuda_graph_jit_source(const cproc_cuda_node *nodes, uint32_t n_nodes, uint32_t n_inputs,
                                 const uint32_t *out_nodes, uint32_t n_outputs, int has_changed, char *dst, size_t cap);

/* ---- dynamic patcher (SURVEY 8 f-2) ---------------------------------------- */
/* The run-time way to build a graph: the RPC tree of stm32f103/mod_bpmodular.c
 * (class/<c>/apply, inst/<node>/state/<k>/get|set, patch/reset, patch/tick) with the
 * instances held as N-wide batches on the device.  Classes: 0 acc, 1 edge, 2 glide
 * (config = div_log), 3 input (config = external stream index; the role gpin has on
 * the microcontroller), 4 pdm (inputs in, dither; config = order | out_shift << 3).  Field names as in the proc_meta tables (cproc.h:107-122).
 * kind: 0 param, 1 state (PARAM / STATE, mod_bpmodular.c:126-127), 2 input, 3 config. */
typedef struct cproc_cuda_patch cproc_cuda_patch;
int  cproc_cuda_patch_class_count(void);
const char *cproc_cuda_patch_class_name(uint32_t cls);
int  cproc_cuda_patch_class_field(uint32_t cls, uint32_t kind, uint32_t k, const char **name);
int  cproc_cuda_patch_open(cproc_cuda_ctx *ctx, uint64_t n_instances, uint32_t n_inputs, uint32_t layout, cproc_cuda_patch **patch);
int  cproc_cuda_patch_close(cproc_cuda_patch *patch);
int  cproc_cuda_patch_reset(cproc_cuda_patch *patch);
int  cproc_cuda_patch_node_count(const cproc_cuda_patch *patch);
/* Returns the new node index (>= 0) or a negative CPROC_CUDA_E* code. */
int  cproc_cuda_patch_apply(cproc_cuda_patch *patch, uint32_t cls, const uint32_t *in_nodes, uint32_t n_in, uint32_t config);
int  cproc_cuda_patch_output(cproc_cuda_patch *patch, uint32_t node);
/* F ticks of every node; io->in [inst][n_inputs][F], io->out the output node's .out.
 * device_buffers != 0: device pointers, asynchronous (cproc_cuda_run_dev). */
int  cproc_cuda_patch_tick(cproc_cuda_patch *patch, uint64_t n_frames, const cproc_cuda_io *io, int device_buffers);
int  cproc_cuda_patch_get(cproc_cuda_patch *patch, uint32_t node, uint32_t kind, uint32_t field, uint64_t instance, uint32_t *value);
int  cproc_cuda_patch_set(cproc_cuda_patch *patch, uint32_t node, uint32_t kind, uint32_t field, uint64_t instance, uint32_t value);
cproc_cuda_batch *cproc_cuda_patch_batch(cproc_cuda_patch *patch);

/* ---- multi-GPU mix bus over NVLink peer memory (SURVEY 8e) ------------------- */
/* One process per GPU.  The only exchange of the path is the shared mix bus: the
 * integer mixes of the shards (io.mix) are summed (square: ORed) and scaled to float
 * once (synth.c:180,194).  Instead of an NCCL all-reduce plus a conversion kernel this
 * is ONE kernel per rank: push the local mix into every peer's bus buffer with stores
 * through the NVLink peer mapping, publish a flag, wait for the peers' flags, add the
 * slots in rank order, write the float bus.  Setup: every rank creates a bus, exports
 * its handle (cproc_cuda_bus_handle_bytes() bytes), the host gathers the handles of
 * all ranks in rank order over its own transport and passes them to _connect.  Every
 * rank must then make the same sequence of _allreduce calls.
 * op: 0 wrap-around sum, 1 OR, 2 float sum in rank order (words are float bits: the float
 * mix of the extension voices; deterministic, scale must be 0).  scale: 0 none, 1 saw (float)(int)x*2^-32, 2 square
 * (float)(unsigned)x*2^-32, 3 grain mix (float)x*2^-7 (out_dev required unless 0). */
typedef struct cproc_cuda_bus cproc_cuda_bus;
int  cproc_cuda_bus_create(cproc_cuda_ctx *ctx, uint64_t max_words, int world, int rank, cproc_cuda_bus **bus);
size_t cproc_cuda_bus_handle_bytes(void);
int  cproc_cuda_bus_handle(cproc_cuda_bus *bus, void *handle);
int  cproc_cuda_bus_connect(cproc_cuda_bus *bus, const void *handles);
int  cproc_cuda_bus_allreduce(cproc_cuda_bus *bus, int32_t *imix_dev, float *out_dev, uint64_t count, uint32_t op, uint32_t scale);
/* Overlapped form: the exchange of block k runs on the bus's own high-priority stream
 * (after everything queued on the context stream so far) while the context stream renders
 * block k+1 into the other mix buffer.  slot 0/1 names the buffer pair; _wait(slot) makes
 * the context stream wait for that slot's last exchange. */
int  cproc_cuda_bus_allreduce_begin(cproc_cuda_bus *bus, uint32_t slot, int32_t *imix_dev, float *out_dev, uint64_t count, uint32_t op, uint32_t scale);
int  cproc_cuda_bus_wait(cproc_cuda_bus *bus, uint32_t slot);
/* The exchange as the tail of the render kernel.  After _attach, cproc_cuda_run_dev on the batch (VOICE_BANK, XVOICE mix, SQUARE_GRAIN_MIX) renders the
 * shard's mix AND exchanges it in the same launch: the blocks that complete a piece of the local mix push it into every
 * peer's bus buffer, the last one publishes the flags.  io.mix / io.out then receive the bus of ALL ranks (reduced integer
 * words / scaled float), like after _allreduce.
 * mode 1: the reduce runs at the end of the same launch -- io.mix / io.out are valid when it completes.
 * mode 2: pipelined -- the reduce of block k runs beside the render of block k+1 (one extra thread block of that launch), or
 *         in cproc_cuda_bus_flush; io.mix / io.out of call k must stay valid until then and are written there.
 * mode 0 (or bus NULL) detaches.  Every rank makes the same sequence of calls. */
int  cproc_cuda_bus_attach(cproc_cuda_bus *bus, cproc_cuda_batch *batch, uint32_t mode);
int  cproc_cuda_bus_flush(cproc_cuda_bus *bus);
int  cproc_cuda_bus_status(cproc_cuda_bus *bus, uint32_t *failed_epoch);
int  cproc_cuda_bus_destroy(cproc_cuda_bus *bus);

/* Integer mix bus -> float, after a multi-GPU all-reduce of the raw mix:
 * VOICE_BANK saw: (float)(int)x * 2^-32 (synth.c:180); square: (float)(unsigned)x
 * * 2^-32 (:194); SQUARE_GRAIN_MIX: (float)x * 2^-7.  Device pointers. */
int  cproc_cuda_mix_to_float(cproc_cuda_batch *b, const void *imix_dev, float *out_dev, uint64_t count);

/* ---- memory + timing helpers (plumbing for C hosts) ---------------------- */
int  cproc_cuda_dev_alloc(cproc_cuda_ctx *ctx, size_t bytes, void **dev);
int  cproc_cuda_dev_free(cproc_cuda_ctx *ctx, void *dev);
int  cproc_cuda_host_alloc(cproc_cuda_ctx *ctx, size_t bytes, void **pinned);
int  cproc_cuda_host_free(cproc_cuda_ctx *ctx, void *pinned);
int  cproc_cuda_memcpy_h2d(cproc_cuda_ctx *ctx, void *dev, const void *host, size_t bytes);
int  cproc_cuda_memcpy_d2h(cproc_cuda_ctx *ctx, void *host, const void *dev, size_t bytes);
int  cproc_cuda_memset(cproc_cuda_ctx *ctx, void *dev, int value, size_t bytes);
/* CUDA-event stopwatch on the context stream. */
int  cproc_cuda_timer_start(cproc_cuda_ctx *ctx);
int  cproc_cuda_timer_stop(cproc_cuda_ctx *ctx, float *elapsed_ms);
/* Tuning knob by name; unknown names and out-of-range values return EINVAL.  Every setting gives
 * the same results (the tests sweep them); the defaults are the measured best on B200.
 *   planar_bulk      0/2  [2]  PLANAR square_grain / pdm / pwm / one-pole / word-clock / generated-graph streams:
 *                              0 = the register-transpose kernel for square_grain and the scalar kernels for the
 *                              others, 2 = tensor-TMA staging; 2 also runs INTERLEAVED square_grain / pdm / one-pole
 *                              four instances per thread
 *   graph_vec4       0/1  [1]  INTERLEAVED generated graphs: four instances per thread (128-bit accesses)
 *   grain_mix2       0..2 [2]  square_grain mix kernel generation
 *   graph_jit        0/1  [1]  generated graphs compiled with NVRTC (0: table-driven kernel, <= 16 nodes)
 *   pdm_ws           0/1  [1]  PDM v2: 1 = producer / consumer kernel under the dynamic (group, time-slice) schedule,
 *                              0 = plain thread-per-bank / thread-per-channel kernels
 *   pdm_tlog         6/7  [7]  PDM v2: log2 of the ticks per producer -> consumer hand-off
 *   pdm_ctas_per_sm [4], pdm_slice_batches [64: work items of 64 x 64 ticks]   PDM v2 dynamic schedule
 *   pdm_planar_bulk  0/2  [2]  PDM v2 PLANAR duty rows: scattered 16-byte stores, tensor-TMA boxes
 *   pdm_v1_chains    1/2  [2]  PDM v1: PRNG chains per lane
 *   pdm_block, pdm_tpb [2: auto; 1 thread per bank when bank_size <= 4; 0 thread per channel], pdm_persist, pdm_warps_per_smsp   plain PDM kernels, PDM v1 schedule
 *   xvoice_mix2      0/1  [1]  XVOICE mix-only render: voice pairs on the packed fp32 pipe (FFMA2) with state tiles in shared
 *                              memory; 0 = the scalar kernel (state through L2 once per 32-frame chunk).  Known deviation of 1:
 *                              it runs the filter on -lp, so where lp + f*bp cancels exactly the state holds lp = -0, not +0
 *   xvoice_mix2_blocks 0..3 [0] its resident blocks per SM (0 = chosen from the voice count)
 *   xvoice_chunk [0 = auto], xvoice_groups 0..8 [0 = one group], xvoice_closed 0/1 [1]
 *                              XVOICE_SCAN: frames per time chunk, variant groups, closed-form zero-state pass
 *   run_graph        0..3 [2]  cproc_cuda_run on small host buffers: staged copies, CUDA graph with copy nodes,
 *                              CUDA graph on pinned staging, direct launches on pinned staging */
int  cproc_cuda_set_option(cproc_cuda_ctx *ctx, const char *name, int64_t value);

#ifdef __cplusplus
}
#endif
#endif /* CPROC_CUDA_H */
