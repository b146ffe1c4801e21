/*
 * xline_b200 -- C ABI of the B200-native `Line.track` particle push.
 *
 * This is the drop-in boundary for the one hot path this library replaces: the
 * reference's element-by-element push
 *
 *     Line.track(p):  for el in self.elements: el.track(p)     xline/line.py:89-95
 *
 * over the element maps in xline/elements.py and xline/be_beamfields/*.py, acting on a
 * particle container with the attributes of xpart's Pyparticles (xline/particles.py:1-6).
 * The reference is pure Python and has no FFI; the entry points below are what a
 * ctypes/cffi binding added to the reference's `Line.track` would call (the stub is in
 * INTEGRATION.md).  Plain pointers and sizes only -- no torch types cross this boundary.
 *
 * Conventions
 *   - every function returns 0 on success, a negative XLB_E* code on failure;
 *     xlb_last_error() returns a thread-local, NUL-terminated description.
 *   - "device" entry points take CUDA device pointers and a cudaStream_t (as void*),
 *     enqueue work on that stream and (unless stated) do not synchronise the device;
 *     "host" entry points take host pointers, perform the H2D/D2H copies themselves and
 *     return when the results are in the host buffers.
 *   - particle state is structure-of-arrays, fp64 / int64, length n, caller-owned.
 *     Lost particles are NOT removed from the arrays (the reference compacts them,
 *     xline/elements.py:420): they keep the coordinates they had at the aperture with
 *     state = 0, at_element = index of the aperture in the Line, at_turn = turn of loss.
 */
#ifndef XLINE_B200_H
#define XLINE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XLB_ABI_VERSION 4

/* error codes */
#define XLB_OK 0
#define XLB_EINVAL (-1)    /* bad argument (null pointer, negative size, bad lattice)  */
#define XLB_ECUDA (-2)     /* CUDA runtime error (message in xlb_last_error)            */
#define XLB_ELATTICE (-3)  /* packed lattice failed validation                          */
#define XLB_ENOGPU (-4)    /* no CUDA device / not an sm_100 class device               */

/* ---------------------------------------------------------------------------------
 * Packed lattice ("flat device lattice buffer": element type tags + fp64 parameters).
 *
 * A lattice is an array of 8-byte words, cut into `n_chunks` chunks of `chunk_words`
 * words (chunk_words even, chunk = unit of one TMA bulk copy into shared memory).  A
 * chunk is a sequence of records; a record starts on an even word (16 B aligned):
 *
 *   word 0  header  = tag (8 bits) | aux << 8 (8 bits) | size << 16 (14 bits, record length
 *                     in 16-byte pairs) | XLB_HDR_* flags (bits 30, 31) |
 *                     (uint64)element_index << 32
 *   word 1  first fp64 parameter (or padding)
 *   word 2..        further parameters, record padded to an even number of words
 *
 * Records never straddle a chunk; every chunk ends with an XLB_T_END_CHUNK record and
 * the last chunk ends with XLB_T_END_TURN instead.  Parameter layout per tag is
 * documented next to the tag.
 *
 * Path length.  `s` advances by the drift lengths only (elements.py:56,72), by the same
 * amount for every particle that stays in the beam.  The fast kernels therefore do no
 * arithmetic on it in the element maps: word 1 of an END_TURN record is the length of the
 * pass it closes (the whole lattice, or one segment of a segmented lattice), added once per
 * pass; and every record at which a particle can be lost (the LIMIT_* tags and the block
 * records) carries `s_here`, the drift lengths from the start of the pass up to the
 * record, added for the particles it removes.  The strict kernels ignore both and keep the
 * reference's per-particle sequential sum.  `element_index` is the position in the reference's
 * `Line.elements` list (what `at_element` reports).  Two encodings exist, selected by
 * XLB_F_STRICT: "fast" (constants pre-folded for FMA-friendly evaluation) and "strict"
 * (raw reference parameters, evaluated in the reference's operation order).
 * --------------------------------------------------------------------------------- */
enum xlb_tag {
  XLB_T_END_TURN = 0,       /* [hdr,length of the pass that ends here]                */
  XLB_T_END_CHUNK = 1,      /* no parameters                                          */
  XLB_T_DRIFT = 2,          /* [hdr,length]                      elements.py:48-56    */
  XLB_T_DRIFT_EXACT = 3,    /* [hdr,length]                      elements.py:64-72    */
  XLB_T_MULTIPOLE = 4,      /* aux=order; [hdr,0] then (kn_i,ks_i) i=order..0
                               fast: kn_i = knl[i]/i!            elements.py:120-156  */
  XLB_T_MULTIPOLE_CURVED = 5, /* aux=order; [hdr,hxl][hyl,length][inv_length,0] then
                               pairs as above                    elements.py:139-154  */
  XLB_T_CAVITY = 6,         /* [hdr,voltage][k=2*pi*f/c, lag_rad] elements.py:239-245 */
  XLB_T_RFMULTIPOLE = 7,    /* aux=order; [hdr,voltage][k,lag_rad] then per order
                               [knl_i,ksl_i][pn_i_rad,ps_i_rad]  elements.py:182-227  */
  XLB_T_XYSHIFT = 8,        /* [hdr,dx][dy,0]                    elements.py:274-276  */
  XLB_T_SROTATION = 9,      /* [hdr,cos][sin,0]                  elements.py:379-390  */
  XLB_T_DIPOLE_EDGE = 10,   /* [hdr,r21][r43,0]                  elements.py:538-548  */
  /* The LIMIT_* records may carry the drift that follows the aperture (pack-time peephole
     Limit* -> Drift): aux bit 4 (XLB_AUX_DRIFT), bit 5 = it is a DriftExact; the drift length
     follows the record's own pairs as [length,0] (LIMIT_POLYGON: in word 3, see there).       */
  XLB_T_LIMIT_RECT = 11,    /* aux bit 0: symmetric box (fast encoding only);
                               [hdr,min_x][max_x,min_y][max_y,s_here] elements.py:401-420 */
  XLB_T_LIMIT_ELLIPSE = 12, /* [hdr,a*a][b*b,1/(a*a)][1/(b*b),s_here] elements.py:429-442 */
  XLB_T_LIMIT_RECT_ELLIPSE = 13, /* [hdr,max_x][max_y,a*a][b*b,1/(a*a)][1/(b*b),s_here]
                                                                 elements.py:453-474  */
  XLB_T_MONITOR = 14,       /* [hdr,0][i64 start,i64 skip][i64 num_stores,i64 min_id]
                               [i64 max_id,i64 rolling][i64 data_offset,0]
                                                                 elements.py:485-527  */
  XLB_T_SAWTOOTH_CAVITY = 15, /* as CAVITY                       elements.py:257-263  */
  XLB_T_BEAMBEAM4D = 16,    /* see xline_b200/lattice.py         beambeam.py:45-82    */
  XLB_T_SPACECHARGE = 17,   /* aux bits 0-3 = profile kind (0 coasting,1 q-Gaussian,2 linear
                               interp,3 cubic spline); aux bit 4/5: the kick is followed by
                               a Drift / DriftExact of length word 1  spacecharge.py  */
  XLB_T_BEAMBEAM6D = 18,    /* [hdr,(double)n_slices] ...        BB6D.py:15-155       */
  /* Polygonal aperture (LimitPolygon; the reference's track raises, so the project defines it).
     Same in both encodings: [hdr,i64 n_edges][s_here,drift_length or 0] then per stored edge
     [y_lo,y_hi][x_lo,slope].  aux bits XLB_AUX_DRIFT / XLB_AUX_DRIFT_EXACT as on the other
     LIMIT_* records (the drift length is word 3, always present).
     The vertices V_k, k = 0..n-1, close into a polygon with edges V_k -> V_(k+1) mod n;
     orientation does not matter, self-intersecting polygons follow the even-odd rule.  For every
     edge with y_k != y_(k+1), (x_lo, y_lo) is the end with the smaller y, y_hi the other end's
     y, and slope = (x_hi - x_lo) / (y_hi - y_lo) in fp64, rounded once at pack time; horizontal
     edges are dropped (they can never be crossed).  A particle at (x, y) crosses an edge iff
     y_lo <= y < y_hi and x < v, where t = y - y_lo; u = t * slope; v = x_lo + u are three
     fp64 operations rounded to nearest with no fused multiply-add.  It is inside iff it crosses
     an odd number of edges, else lost: NaN / inf coordinates are lost; on an axis-aligned
     boundary points of the left and bottom edges are inside, of the right and top edges outside.
     Every implementation of the predicate gives bit-identical loss flags.  A lattice with these
     records carries XLB_F_POLYGONS.  Added without an ABI version change: a library that
     predates the tag refuses the lattice in xlb_lattice_validate ("unknown tag").           */
  XLB_T_LIMIT_POLYGON = 19,
  /* Radiating multipole (DESIGN.md §4.9): a Multipole of length L > 0 on a line tracked with
     synchrotron radiation.  Fast encoding only.  aux = order;
       [hdr,i64 mode (1 mean, 2 quantum)][L,1/L][K_e,hbar_c][alpha,u64 seed]
       then the element's own MULTIPOLE or MULTIPOLE_CURVED record, header word included, exactly
       as it is packed on its own (hxl, hyl come from there; 0 for the straight one).
     K_e = e^2/(4 pi eps0) and hbar_c in eV m, alpha the fine-structure constant: taken at pack
     time, nothing physical is compiled into the kernel.  q0, mass0, p0c come from the call.
     Map, with (dpx_f, dpy_f) the Horner polynomial of knl/ksl (k0l included) at the element's
     (x, y) -- the field part of the kick, without the hxl/hyl reference-frame terms:
       kappa = sqrt(dpx_f^2 + dpy_f^2) / ((1 + delta) L),  l_h = (L + hxl x - hyl y) / 2;
       1. radiate over l_h;  2. the multipole map of the embedded record, unchanged;
       3. radiate over l_h with kappa recomputed from the new delta (x, y and the field unchanged).
     Radiating an energy dE < 0 (P = (1+delta) p0c, E = sqrt(P^2 + m^2), gamma = E/m, beta = P/E, with
     m^2 = (energy0 - p0c)(energy0 + p0c) from the call's reference particle -- for a 6 GeV electron
     the rounding of energy0 leaves m, and so the loss, uncertain at the 1e-8 level):
       Pyparticles.add_to_energy(dE) as Cavity does (delta, rpp, rvv, zeta rvv'/rvv), then px and
       py times (1+delta')/(1+delta): the photon leaves along the direction of motion.
       mean:    dE = -(2/3) q0^2 K_e beta^3 gamma^4 kappa^2 l_h;
       quantum: k ~ Poisson(nbar), nbar = (5/(2 sqrt 3)) q0^2 alpha gamma kappa l_h, k <= 255;
                dE = -u_c sum_{i=1..k} x_i, u_c = (3/2) hbar_c gamma^3 kappa, x_i = F^-1(U_i) of
                the photon-number spectrum dN/dx ~ int_x^inf K_5/3 (csrc/synrad_table.inc).
       The quantum mode's expected loss is (2/3) q0^2 K_e gamma^4 kappa^2 l_h: the mean mode's up to
       the factor beta^3 = 1 - O(1/gamma^2).  A half with kappa == 0 (mean) or k == 0 (quantum)
       leaves the particle untouched.
     Random numbers: Philox4x32-10, key (lo32(seed), hi32(seed)), counter (lo32(particle_id),
       hi32(particle_id), lo32(turn), element << 8 | half << 7 | j), where turn = the particle's
       at_turn at the element (stored value + turns of this call), element = the record's element
       index + element_index_offset (< 2^24), half 0 / 1 (entrance / exit).  Output words
       r0..r3 of call j give the uniforms 2j (from w = r1 2^32 + r0) and 2j + 1 (w = r3 2^32 + r2),
       U = ((w >> 11) + 0.5) 2^-53 in (0, 1).  Uniform 0 gives k: the smallest i with U <= C_i,
       C_0 = p_0 = exp(-nbar), p_i = p_(i-1) nbar / i, C_i = C_(i-1) + p_i (capped at 255; never
       reached for nbar below ~100).  Uniforms 1..k give x_1..x_k.
     Reproducibility: every draw is a function of (seed, particle_id, turn, element, half) alone,
       so results are bitwise independent of particles per thread, threads per block,
       turns_per_launch, the work queue, survivor compaction and the rest of the batch; T1 turns
       then T2 turns equal T1 + T2 turns.
     A lattice with these records carries XLB_F_RADIATION.  Refused (XLB_ELATTICE): a strict
     lattice, beam-field records, more than 2^24 elements.  Refused (XLB_EINVAL) at tracking
     time: a chi column (multi-species beams), element_index_offset + n_elements > 2^24, and the
     tangent map.  Added without an ABI version change: a library that predates the tag refuses
     the lattice in xlb_lattice_validate ("unknown tag").                                       */
  XLB_T_MULTIPOLE_RAD = 20,
  XLB_T__COUNT = 21,
  /* Exciter (DESIGN.md §4.11): a thin multipole whose strength is read, per particle, from a sampled
     waveform by turn and arrival time -- AC dipole, power-converter ripple, transverse excitation.
     It lies outside the contiguous single-element tags 0 .. XLB_T__COUNT-1, which keep their meaning
     for code written against them (a scan that refuses tag >= XLB_T__COUNT still refuses it); 0x40
     has bit 7 clear, so none of the block-family masks (tag & 0xc0 == 0x80, tag & 0xe0) match it.
     0x40 is the one valid tag in 0x40 .. 0x7f; every other value there is an unknown tag.  Fast
     encoding only.  aux = order;
       [hdr,A][B,i64 start_turn][i64 n_samples,i64 data_offset] then (kn_i,ks_i) i=order..0
     with kn_i = knl[i]/i! as in MULTIPOLE, A = sampling_frequency/frev and B = sampling_frequency/c
     taken at pack time.  The samples are n_samples fp64 words at words[data_offset ..], in the data
     region after the chunks (see xlb_lattice_t::n_words): data_offset is an absolute word index.
     Map, for a particle at turn T (its at_turn: the stored value + the turns of this call, as BeamMonitor
     takes it) with beta0 from the call's reference particle:
       t = (double)(T - start_turn)                 exact for |T - start_turn| < 2^53
       u = t*A - (zeta*B)/beta0                      the products, the quotient and the difference
       v = floor(u + 0.5)                            each rounded to nearest, no fused multiply-add
                                                     (a quotient off by an ulp where |zeta*B| < 2^-960
                                                     leaves u unchanged: the kernel's reciprocal form)
       s = samples[(int64)v] if 0 <= v < n_samples, else 0 (no kick; a NaN or infinite zeta gives none)
       (Px, Py) = the Horner polynomial of knl/ksl at (x, y), as MULTIPOLE (straight: no hxl/hyl)
       px <- px - chi*(s*Px),  py <- py + chi*(s*Py)
     The index is a fixed sequence of IEEE operations, so every implementation picks the same sample;
     rounding to nearest makes a particle with |zeta| < C/2 read the sample of its own turn when
     sampling_frequency == frev.  A lattice with these records carries XLB_F_EXCITER.  Refused: a
     strict or segmented lattice (XLB_ELATTICE; a segment's kernel sees the segment's first chunk as
     word 0) and the tangent and envelope entry points (XLB_EINVAL: a
     turn-dependent map has no closed orbit).  Added without an ABI version change: a library that
     predates the tag refuses the lattice in xlb_lattice_validate ("unknown tag").                */
  XLB_T_EXCITER = 0x40,
  /* Fused thin multipole -> [aperture] -> [drift] records (pack-time peephole).  The tag
     has bit 7 set and describes the block: bits 0-1 aperture kind (0 none, 1 symmetric
     rect, 2 rect, 3 ellipse), bit 2 curved multipole, bit 3 drift present, bit 4 that drift
     is a DriftExact.  aux=order;
     [hdr,drift_length][i64 aperture_element_index,s_here] (kn_i,ks_i) i=order..0
     [hxl,hyl][length,1/length] if curved (header bit XLB_HDR_HX_ONLY: hyl == 0, fast encoding)
     [min_x,max_x][min_y,max_y] (rect) or [a*a,b*b][1/(a*a),1/(b*b)] (ellipse)            */
  XLB_T_THIN_BLOCK = 0x80,
  /* Merged block (fast encoding only): two co-located thin multipoles K1, K2 evaluated as ONE
     multipole with summed coefficients -- [K1][A1][K2][A2][drift] of the Line, where thin kicks
     leave x, y untouched so both aperture tests are unaffected.  Tag = 0xA0 | the thin-block
     bits (A2 kind, K2 curved, drift, exact).  aux = merged order;
     [hdr,drift_length][i64 a1_index | a2_index << 32, i64 k1_order | has_a1 << 8]
     merged (kn_i,ks_i) i=order..0  [hxl,hyl][length,1/length][knl0,ksl0 of K2] if curved
     [a*a,b*b][1/(a*a),1/(b*b)] if has_a1 (A1 is an ellipse)  A2 limits as above
     K1's own (kn_i,ks_i) i=k1_order..0 (re-evaluated only for particles lost at A1)
     [s_here,0]                                                                            */
  XLB_T_MERGED_BLOCK = 0xA0,
  /* Dipole edge followed by a drift: tag = 0xC0 | drift << 3 | exact << 4;
     [hdr,drift_length][r21,r43]                              elements.py:538-548, 48-72   */
  XLB_T_EDGE_BLOCK = 0xC0
};

/* Header bit 31, fast encoding, curved block records only: the multipole's hyl is exactly 0 (a
   horizontal bend).  The kernel then leaves the hyl terms of elements.py:139-154 out -- exact
   zeros for every finite y -- which saves 6 of the 14 FP64 instructions of the curved kick.
   Optional: a packer that never sets it gets the general formula.                          */
#define XLB_HDR_HX_ONLY 0x80000000u
/* aux bits of the LIMIT_* and SPACECHARGE records: a drift fused into the record              */
#define XLB_AUX_DRIFT 0x10
#define XLB_AUX_DRIFT_EXACT 0x20
/* Header bit 30, merged block records: the block has an aperture A1 between its two kicks (the
   same fact as bit 8 of the record's second i64; the header copy is warp-uniform in the kernel).
   Mandatory on merged blocks with an A1.                                                    */
#define XLB_HDR_HAS_A1 0x40000000u

typedef struct xlb_lattice {
  const uint64_t *words; /* n_chunks * chunk_words words, then the data region (if any)  */
  /* n_chunks * chunk_words, plus the words of the data region on a lattice flagged XLB_F_EXCITER:
     n_data_words fp64 words after the last chunk that hold the exciters' waveforms.  The kernels
     stream the chunks only; they read the data region through the read-only data path.          */
  int64_t n_words;
  int32_t chunk_words;   /* even, 16 <= chunk_words*8 <= 96 KiB                         */
  int32_t n_chunks;
  int32_t n_elements;    /* length of the reference Line (size of loss tallies)         */
  uint32_t flags;        /* XLB_F_* below                                               */
  /* Segmented lattice (fast encoding of lattices with BeamBeam6D lenses): the chunks form
     n_segments consecutive groups, each terminated by END_TURN, that are executed one after
     the other every turn -- XLB_SEG_MAIN groups by the tracking kernel, XLB_SEG_BB6D groups
     (one chunk holding one BEAMBEAM6D record) by the stand-alone 6D-lens kernel.  The last
     group is a MAIN group (possibly empty); it is the one that counts the turn.  `segments`
     is a HOST array of n_segments triples {first_chunk, n_chunks, kind}, also when `words`
     is device memory.  n_segments == 0: the whole lattice is one MAIN group.            */
  int32_t n_segments;
  const int32_t *segments;
} xlb_lattice_t;

#define XLB_SEG_MAIN 0
#define XLB_SEG_BB6D 1

#define XLB_F_STRICT 1u      /* lattice encoded for / kernel evaluates in the reference's
                                operation order without FMA contraction                 */
#define XLB_F_BEAMFIELDS 2u  /* the MAIN groups contain BEAMBEAM4D/6D or SPACECHARGE records */
#define XLB_F_BB6D 4u        /* lattice contains BEAMBEAM6D records: in MAIN groups (then
                                BEAMFIELDS is set too and the kernels that carry the 6D
                                lens are used) or in XLB_SEG_BB6D groups                */
#define XLB_F_LOW_ORDER 8u   /* every MULTIPOLE / block record has order (aux) <= 3: the
                                kernels with a straight-line Horner evaluation may be used
                                (checked by xlb_lattice_validate; optional, never required) */
#define XLB_F_POLYGONS 16u   /* the lattice holds LIMIT_POLYGON records (mandatory: checked by
                                xlb_lattice_validate; the kernels that can track them are used) */
#define XLB_F_RADIATION 32u  /* the lattice holds MULTIPOLE_RAD records (mandatory: checked by
                                xlb_lattice_validate; only the one-species thin-lens fast
                                kernels carry the case)                                  */
#define XLB_F_EXCITER 64u    /* the lattice holds EXCITER records (mandatory: checked by
                                xlb_lattice_validate, which accepts a data region after the chunks
                                only with this flag; the kernels that carry the case are used) */
#define XLB_RAD_MEAN 1
#define XLB_RAD_QUANTUM 2
#define XLB_RAD_MAX_ELEMENTS (1 << 24)

/* Particle set, mirrors the attributes the reference's elements read and write
 * (SURVEY.md §8a row a2).  All arrays have length n.  chi and charge_ratio may be NULL
 * (treated as 1.0).  chi == NULL is the fast case: one species, the reference's default -- the
 * kernels compiled without a chi register are used (4 particles per thread instead of 3);
 * xlb_track_host passes NULL on by itself when the host chi column is all ones.
 * s, particle_id, at_element, at_turn may NOT be NULL. */
typedef struct xlb_particles {
  int64_t n;
  double *x, *px, *y, *py, *zeta, *delta, *rpp, *rvv, *s;
  const double *chi, *charge_ratio;
  int64_t *state, *at_element, *at_turn;
  const int64_t *particle_id;
  double q0, mass0, p0c, beta0, gamma0, energy0; /* reference particle                  */
} xlb_particles_t;

typedef struct xlb_track_options {
  int32_t num_turns;         /* >= 0                                                     */
  int32_t particles_per_thread; /* 0 = default (4 for thin-lens lattices with chi == NULL, 3
                                   with a chi column or strict, 2 for beam-field lattices;
                                   fewer when the beam would not fill the GPU); 1..4       */
  int32_t threads_per_block;    /* 0 = default (128; 256 for beam-field lattices at 1-2
                                   particles/thread); multiple of 32, <= the variant's
                                   launch bound                                            */
  int32_t turns_per_launch;  /* > 0: survivors are re-compacted (warp-ballot stream
                                compaction) between launches of this many turns; 0 =
                                automatic (one launch up to 150 turns, else launches of 100
                                turns); < 0 = all turns in one launch                      */
  int64_t *loss_tally;       /* optional [n_elements] int64 counters, incremented per
                                element where a particle was lost (same memory space as
                                the particle arrays)                                     */
  double *monitor_data;      /* optional BeamMonitor storage (fp64 words), see
                                XLB_T_MONITOR; same memory space as the particles        */
  int64_t monitor_words;     /* capacity of monitor_data in fp64 words                   */
  double compact_threshold;  /* re-compact when lost/active exceeds this (default 1/128) */
  int32_t turns_per_item;    /* granularity of the device-side work queue: a launch of more
                                turns than this, over more particle blocks than there are SMs,
                                runs persistent CTAs that pull (particle block, turn segment)
                                items.  0 = automatic (one turn, or as many as stream 16
                                lattice chunks), < 0 = off                                */
  int32_t flags;             /* XLB_OPT_* below                                          */
  double *trace;             /* optional element-by-element trace, [n_elements][6][trace_particles]
                                fp64 (x px y py zeta delta after every element for the first
                                trace_particles particle slots; the device form of
                                Line.track_elem_by_elem, xline/line.py:97-108).  Needs
                                num_turns == 1 and a lattice packed without record fusing     */
  int64_t trace_particles;
  int64_t element_index_offset; /* added to the element index recorded in at_element (not to the
                                loss-tally index): a caller that pushes the elements of a Line
                                one call at a time -- el.track(p) in a loop, the reference's
                                track_elem_by_elem (xline/line.py:97-108) -- passes the position
                                of the element in that Line                                 */
} xlb_track_options_t;

#define XLB_OPT_NO_TURN_COUNT 1 /* do not advance at_turn at the end of the lattice: the call is
                                   one element (or a part) of a turn, like the reference's
                                   el.track(p), which never touches the turn counter          */

/* Statistics of the last xlb_track_* call on this thread. */
typedef struct xlb_track_stats {
  int64_t n_alive_in, n_alive_out;
  int32_t kernel_launches;   /* tracking-kernel launches                                 */
  int32_t compactions;       /* compaction-kernel launches                               */
  int32_t regs_per_thread, smem_bytes, blocks, threads; /* last tracking launch          */
  float kernel_ms;           /* CUDA-event time of the tracking kernels (host entry point
                                and xlb_track_device_timed only)                         */
} xlb_track_stats_t;

int xlb_abi_version(void);
const char *xlb_last_error(void);

/* Validates a packed lattice held in HOST memory (record structure, tags, chunking). */
int xlb_lattice_validate(const xlb_lattice_t *host_lattice);

/* The hot path, device pointers.  Replaces the loop of xline/line.py:89-95 repeated
 * opts->num_turns times.  lattice->words, all particle arrays, opts->loss_tally and
 * opts->monitor_data are DEVICE pointers.  `stream` is a cudaStream_t.  Synchronises the
 * stream only when turns_per_launch splits the job (to read the survivor count). */
int xlb_track_device(const xlb_lattice_t *lattice, xlb_particles_t *particles,
                     const xlb_track_options_t *opts, void *stream);

/* Same, but brackets the tracking kernels with CUDA events on `stream`, synchronises and
 * reports kernel_ms through xlb_get_stats(). */
int xlb_track_device_timed(const xlb_lattice_t *lattice, xlb_particles_t *particles,
                           const xlb_track_options_t *opts, void *stream);

/* The hot path, HOST pointers (what a NumPy-holding caller such as the reference's own
 * Line.track would bind): copies lattice + particle columns to the current device, tracks,
 * copies the particle columns (and tallies / monitor data) back.  Blocking. */
int xlb_track_host(const xlb_lattice_t *host_lattice, xlb_particles_t *host_particles,
                   const xlb_track_options_t *opts);

int xlb_get_stats(xlb_track_stats_t *out);

/* Stream compaction of survivors: writes the indices i with state[i]==1, in increasing
 * order, to idx_out (device, capacity n) and their count to *n_out (device).  Warp-ballot
 * prefix scan; deterministic.  Used internally between launches and exposed for the host
 * container's remove_lost_particles(). */
int xlb_compact_alive_device(const int64_t *state, int64_t n, int32_t *idx_out,
                             int32_t *n_out, void *stream);

/* ---------------------------------------------------------------------------------
 * Beam moments (DESIGN.md §4.6): the number of particles and the first and second moments of
 * (x, px, y, py, zeta, delta) over the surviving beam, taken on the device.
 *
 * A particle counts iff state == 1 and its six coordinates are all finite; alive particles with
 * a non-finite coordinate are counted apart.  A store is XLB_MOMENT_WORDS fp64 words:
 *   [0] n   [1] n_nonfinite   then XLB_MOMENT_PAIRS (hi, lo) pairs: the 6 sums  Σu  in the
 *   order x px y py zeta delta (pair 0..5), then the 21 sums  Σu·v  for u <= v, upper triangle in
 *   row-major order: xx xpx xy xpy xzeta xdelta pxpx pxy ... deltadelta (pair 6..26).
 * Each product u·v is taken exactly (TwoProduct with an FMA), so each sum is a sum of exact
 * terms, accumulated in double-double.
 * Accuracy: |hi + lo - exact sum| <= 3·2^-106·ceil(log2 n)·Σ|terms| (n = the particle count of
 *   the call), which is <= 2^-100·Σ|terms| up to n = 2^21.
 * Reproducibility: the summation order is a fixed binary tree over the slot index 0..n-1, so a
 *   store is bitwise independent of the kernel family, the particles per thread, the threads per
 *   block, turns_per_launch, turns_per_item, survivor compaction and the launch-length schedule.
 * --------------------------------------------------------------------------------- */
#define XLB_MOMENT_WORDS 56
#define XLB_MOMENT_PAIRS 27
#define XLB_MOMENT_FIRST 2  /* word of the first pair (Σx hi) */

/* Store turns of one tracking call: store k is taken after t_k = start + k·skip turns of the
 * call, for k < num_stores and t_k <= num_turns (t = 0 is the beam before the first turn, at the
 * start of the line).  Stores with t_k > num_turns are not written; every other store is, also
 * when the beam is already empty.  num_stores, start >= 0, skip >= 1. */
typedef struct xlb_moments_spec {
  int64_t num_stores;
  int64_t start;
  int64_t skip;
} xlb_moments_spec_t;

/* One snapshot of the particles (device pointers; x..delta and state are read) into the
 * XLB_MOMENT_WORDS words at `out` (device).  Enqueued on `stream`, no synchronisation. */
int xlb_beam_moments_device(const xlb_particles_t *particles, double *out, void *stream);

/* xlb_track_device, plus the stores of `spec` into out[k·XLB_MOMENT_WORDS ..] (device, capacity
 * spec->num_stores stores).  Launches are cut so that one ends on every store turn, and the
 * reduction runs on the stream after it: the particles are tracked exactly as without stores.
 * Like a job split by turns_per_launch, it synchronises the stream between launches.
 * Strict, beam-field and segmented lattices; a trace is refused (XLB_EINVAL). */
int xlb_track_device_moments(const xlb_lattice_t *lattice, xlb_particles_t *particles,
                             const xlb_track_options_t *opts, const xlb_moments_spec_t *spec,
                             double *out, void *stream);

/* ---------------------------------------------------------------------------------
 * NAFF tunes (DESIGN.md §4.7): the frequency and amplitude of the largest spectral line of
 * turn-by-turn signals, for tune footprints and frequency maps.
 *
 * A signal is T = num_turns samples u_t (and optionally pu_t), t = 0 .. T-1.  The analysed z_t:
 *   complex (pu given):  z_t = u_t/√β - i·(α·u_t + β·pu_t)/√β  (√(2J)·e^{+iφ_t} for linear motion
 *                        at a point with Twiss β > 0, α: the peak sits at +ν, ν in [0, 1));
 *                        β = 1, α = 0 gives x - i·px;
 *   real (pu NULL):      z_t = u_t, ν in [0, 1/2]; β and α are ignored.
 * 1. z_t <- z_t - (1/T)·Σ z_t.
 * 2. Hann window w_t = 1 - cos(2πt/T)  (Σ w_t = T).
 * 3. Z(ν) = Σ_t w_t·z_t·e^{-2πiν(t - T/2)}  (the centred phase changes the phase of Z only).
 * 4. Coarse peak: M = the smallest power of two >= T; k = argmax |Z(k/M)| (zero-padded DFT) over
 *    k = 1 .. M-1 (complex) or k = 1 .. M/2 (real), the lowest k on ties.
 * 5. The root ν of D(ν) = Re(conj(Z)·Z') (Z', Z'' derivatives in ν) in [(k-1)/M, (k+1)/M]:
 *    Newton from k/M, D'(ν) = |Z'|² + Re(conj(Z)·Z''), with a bisection safeguard (a step that
 *    leaves the bracket, or D' >= 0, bisects; D > 0 raises the lower end, else the upper one).
 *    It stops when a step is below 1e-15, when D = 0 with D' < 0, or after 40 steps (D = 0 with
 *    D' >= 0 -- e.g. ν = 1/2 between a real signal's line and its mirror image -- bisects).
 * 6. tune = ν folded into the range above (the brackets of k = M-1 and k = M/2 reach past
 *    it): ν - 1 for a complex ν >= 1, 1 - ν for a real ν > 1/2, both exact;  amplitude = |Z|/Σ w_t at the last evaluation (|Z| is stationary there), which is
 *    √(2J) for a linear particle in normalised coordinates.
 * 7. A non-finite sample (a particle lost inside the window, an id never stored): tune and
 *    amplitude NaN.  z = 0 after step 1: tune NaN, amplitude 0.
 * Accuracy: a pure complex tone is recovered to ~1e-11 at T ~ 1000 (real tones ~1e-9: the mirror
 *   line at -ν leaks through the window; within ~1/T of 0 or 1/2 the two lines merge and the real
 *   tune comes out near 0 or 1/2); most of the remaining error is leakage from the
 *   subtracted mean.  The device computes the same root of D as a float64 evaluation of the
 *   steps above to ~1e-12 (1e-12 relative in amplitude) unless the two largest coarse bins are
 *   within ~1e-9 of each other.
 * Reproducibility: every sum runs in an order fixed by t alone, so a signal's tune and amplitude
 *   are bitwise independent of n, its position in the batch, the row stride and the launch shape.
 * --------------------------------------------------------------------------------- */
#define XLB_NAFF_MIN_TURNS 64
#define XLB_NAFF_MAX_TURNS 8192

/* NAFF of the n signals j = 0 .. n-1 of a turn-major slab (device pointers): sample t of signal
 * j at u[t·stride + j] and pu[t·stride + j] (the layout of a BeamMonitor field), pu NULL for real
 * signals.  Writes tune_out[j] and amplitude_out[j].  Enqueued on `stream`, no synchronisation.
 * XLB_EINVAL for n < 0, num_turns outside [XLB_NAFF_MIN_TURNS, XLB_NAFF_MAX_TURNS], stride < n,
 * a null pointer with n > 0, or (pu given) β not (finite and > 0) or α not finite.  n = 0: no-op. */
int xlb_naff_device(const double *u, const double *pu, int64_t n, int64_t num_turns, int64_t stride,
                    double beta, double alpha, double *tune_out, double *amplitude_out, void *stream);

/* ---------------------------------------------------------------------------------
 * Tangent map (DESIGN.md §4.8): particles tracked as xlb_track_device tracks them, each carrying
 * its Jacobian  J = dz/dz0  over z = (x, px, y, py, zeta, delta), for chaos indicators, closed
 * orbits and one-turn matrices of the tracked map itself.
 *
 * Lattice: one record per element -- no block records (tags >= 0x80), no segments, the fast
 *   encoding (XLB_F_STRICT clear); BEAMBEAM6D and EXCITER are refused.  MONITOR records are the identity and
 *   store nothing.  rpp and rvv are functions of delta throughout.
 * Layout: jac[i*36 + r*6 + c] = dz_r/dz0_c of particle i (row-major 6x6, r, c in the order of z);
 *   the caller initialises it (the identity for a fresh start).  The true Jacobian is
 *   jac[i] * 2^log2_scale[i].
 * Per turn: J <- J_elem(z before the element) . J for every element; at the end of every turn of a
 *   surviving particle, with m = max|J|: if m > 2^512, J <- J * 2^-ilogb(m) and
 *   log2_scale += ilogb(m) (exact: the result does not depend on when it happens), then
 *     fli <- max(fli, log10 ||J||_F + log2_scale * log10 2).
 *   The caller initialises fli (log10 sqrt(6), the identity's, for a fresh start).
 * Losses: state, at_element, at_turn, s and the loss tally as xlb_track_device; a lost particle's
 *   jac, log2_scale and fli are written where it was lost and not touched again.  Particles with
 *   state != 1 at the call are left alone.
 * Reproducibility: one particle per thread with nothing shared, so results are bitwise independent
 *   of n, the particle's slot and threads_per_block; T1 turns then T2 turns equal T1 + T2 turns.
 * Options: num_turns, loss_tally, flags, element_index_offset and threads_per_block (0 = 128, a
 *   multiple of 32 <= 256) are used; particles_per_thread must be 0 or 1; trace is refused.
 * One launch, enqueued on `stream`; the lattice words are read back to the host once per call to
 *   check the tags (a stream synchronisation).  XLB_EINVAL for the refusals above (the message names
 *   the element) and a null jac / log2_scale / fli with n > 0.
 * --------------------------------------------------------------------------------- */
#define XLB_TANGENT_SCALE_LOG2 512  /* the overflow guard's threshold, 2^512 */
#define XLB_TANGENT_MAX_THREADS 256

int xlb_track_tangent_device(const xlb_lattice_t *lattice, xlb_particles_t *particles,
                             const xlb_track_options_t *opts, double *jac /*[n][6][6]*/, int64_t *log2_scale,
                             double *fli, void *stream);

/* Tangent map with radiation (DESIGN.md §4.10): xlb_track_tangent_device, same contract, on a lattice
 * that may also hold XLB_T_MULTIPOLE_RAD records -- every one of them in mean mode (a quantum record is
 * XLB_EINVAL naming the element: the random map has no tangent).  The checks on a radiating lattice
 * are those of xlb_track_device (one species, no beam fields, element indices < 2^24).  A mean-mode
 * half with kappa == 0 is the identity; otherwise, with W = dE of the half (< 0) as a function of
 * (x, y, delta) through fl^2 (never fl: smooth where the field vanishes) and l_h:
 *   J <- J_h J,  J_h = d(add_to_energy(W), then px, py times (1+delta')/(1+delta)) / dz,
 * so the half is a row update of the delta, zeta, px and py rows.  A lattice without radiating
 * records gives the results of xlb_track_tangent_device bit for bit.                            */
int xlb_track_tangent_radiation_device(const xlb_lattice_t *lattice, xlb_particles_t *particles,
                                       const xlb_track_options_t *opts, double *jac /*[n][6][6]*/,
                                       int64_t *log2_scale, double *fli, void *stream);

/* Beam envelope (DESIGN.md §4.10): particles tracked as xlb_track_tangent_radiation_device tracks
 * them (same lattice checks, options, losses and reproducibility), each carrying a 6x6 second moment
 * Sigma (cov[i*36 + r*6 + c], row-major, symmetric, caller-initialised) and the energy it lost.
 *   Every element: Sigma <- J_e Sigma J_e^T with J_e the element's Jacobian at the state before it.
 *   Every radiating half (mean mode, kappa != 0) adds the variance of the quantum mode's loss in
 *     that half linearised about the mean-mode orbit:  Sigma += V_h g g^T,
 *     V_h = nbar (11/27) u_c^2 (eV^2; nbar, u_c as in the quantum map of XLB_T_MULTIPOLE_RAD, from the
 *     record's K_e, hbar_c, alpha), g = dz_after/dW = (0, px' , 0, py', zeta', delta') of the half's
 *     energy change;  and energy_loss[i] -= W (eV).
 *   At the end of every turn of a surviving particle Sigma <- (Sigma + Sigma^T)/2.
 * A lost particle's Sigma and energy_loss are written where it was lost.  On a lattice without
 * radiating records Sigma is transported without diffusion: J Sigma0 J^T of the same particle's
 * tangent map.  XLB_EINVAL for the refusals of the tangent map and a null cov / energy_loss with
 * n > 0.                                                                                          */
int xlb_track_envelope_device(const xlb_lattice_t *lattice, xlb_particles_t *particles,
                              const xlb_track_options_t *opts, double *cov /*[n][6][6]*/,
                              double *energy_loss /*[n]*/, void *stream);

/* Register-resident independent-DFMA-chain microbenchmark: the measured FP64 pipe peak of
 * the current device in FLOP/s (2 flops per DFMA), best of `repeats`.  The roofline
 * denominator of bench.py (MEASURED_PEAKS.json has no FP64 entry). */
int xlb_measure_fp64_peak(int repeats, double *flops_out, double *ms_out);

/* Single-warp DFMA timing: cycles per DFMA with 1, 2, 4 and 8 independent dependent chains
 * (cycles_per_dfma[0..3]); the first is the dependent-issue latency of the FP64 pipe. */
int xlb_measure_dfma_latency(double *cycles_per_dfma, int n);

/* Device self-test of the strict kernels' division sequences (csrc/track_impl.cuh: reciprocal
 * from the record or the constant table + FMA remainder corrections in place of the IEEE
 * division subroutine; the reference divides at xline/elements.py:130-134, 143-144, 436):
 * every quotient is compared bit for bit with the device's own a / b.  mode 0: integer divisors
 * 1..255 (the Horner step), mode 1: arbitrary positive divisors (`length`, a*a, b*b).  Dividends:
 * random sign and mantissa, exponents uniform in 2^+-exponent_span, every 16th next to a
 * rounding midpoint of the quotient.  *mismatches must come back 0. */
int xlb_selftest_exact_division(const double *divisors, int n_divisors, int mode,
                                int samples_per_thread, uint64_t seed, int exponent_span,
                                uint64_t *mismatches, uint64_t *samples);

/* Number of tracking-kernel variants compiled in, and a description of variant i
 * ("fast/ppt2/lean", ...) with its register count -- build introspection for tests. */
int xlb_kernel_variant_count(void);
int xlb_kernel_variant_info(int i, char *name, int name_len, int *regs, int *max_threads);

#ifdef __cplusplus
}
#endif
#endif /* XLINE_B200_H */
