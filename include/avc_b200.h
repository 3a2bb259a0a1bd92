/*
 * avc_b200.h -- C ABI of libavc_b200.so, the sm_100a kernel library behind the drop-in
 * model classes in autoformer_b200/ (factory.AutoVC / LstmDV / melgan Generator ...).
 *
 * The reference (achyun/Autoformer) has no FFI of its own: its boundary is the Python
 * nn.Module surface (SURVEY.md 8b).  Each entry point below replaces the torch.nn calls the
 * reference makes on the conversion forward path; the citation names the reference lines
 * whose arithmetic the entry point performs.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless said otherwise
 *   - the caller owns every buffer (incl. scratch); the library never allocates device memory
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no host sync inside
 *   - return 0 on success, negative on error; avc_last_error() gives the text (thread local)
 *   - activations are channels-last:  [utterance][frame][channel], channel contiguous
 *   - dtype: 0 = fp32 storage, TF32 tensor-core operands, fp32 accumulate
 *            1 = bf16 storage and operands, fp32 accumulate
 *            2 = "split bf16" (fp32-grade): every fp32 value v is stored as two bf16 channels
 *                hi = bf16(v), lo = bf16(v - hi) in a buffer of 2C channels laid out [hi(0..C) | lo(0..C)];
 *                a product a*w is evaluated as a_hi*w_hi + a_lo*w_hi + a_hi*w_lo by K-concatenating the three
 *                terms into one bf16 tensor-core GEMM (error ~2^-16 instead of TF32's 2^-11, 1.5x the MMA work).
 *                For avc_conv_gemm this is expressed with dtype = 1 and two sources over the same buffer
 *                (source 0: all 2C channels against [w_hi|w_hi]; source 1: the first C channels against w_lo);
 *                out_dtype = 2 makes the epilogue write the split format.
 */
#ifndef AVC_B200_H_
#define AVC_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define AVC_DTYPE_TF32 0
#define AVC_DTYPE_BF16 1
#define AVC_DTYPE_BF16X3 2
#define AVC_DTYPE_F16 3 /* fp16 storage and operands, fp32 accumulate.  "fp16x2" precision: activations are single
                           fp16 values (2^-12 relative), every weight is two fp16 terms w_hi + w_lo (exact to ~2^-22), and a
                           product is a*w_hi + a*w_lo -- two MMA passes instead of the three of dtype 2, end-to-end
                           error ~3e-4 on AutoVC (scripts/precision_study.py).  avc_conv_gemm: two sources over the
                           same buffer against [w_hi | w_lo]; avc_lstm_seq: w = [w_hi | w_lo] like dtype 2. */

#define AVC_ACT_NONE 0
#define AVC_ACT_RELU 1
#define AVC_ACT_TANH 2
#define AVC_ACT_LRELU 3 /* slope 0.2, melgan/modules.py:75,100,120 */
#define AVC_ACT_GELU 4  /* exact erf GELU, nn.GELU() default, factory/MLPMixer.py:19 */
#define AVC_ACT_LOG10_CLAMP 5 /* log10(max(v, 1e-5)), melgan/modules.py:67-68 (Audio2Mel) */

int avc_version(void);
const char* avc_last_error(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
long long avc_launch_count(void);

/*
 * Implicit-GEMM convolution / dense GEMM on the tcgen05 tensor cores (TMA-fed, TMEM accumulators).
 *
 *   v[b, t, n]   = bias[n] + sum_s sum_k sum_c  W[n, (s,k,c)] * A_s[b, tap_t0_s + t + k*tap_dt_s, c]  (+ residual)
 *   out_raw      = v                 (operand format, no halo)              -- optional
 *   out, out2    = act(v)            (operand format with halo / exact fp32) -- optional
 *
 * Replaces: nn.Conv1d + nn.BatchNorm1d(eval) + relu/tanh  (factory/AutoVC.py:26-41,50-51,79-94,104-108,
 * 127-179; factory/Norm.py:21-37), nn.Linear (factory/Norm.py:40-50, factory/AutoVC.py:98,112),
 * the LSTM input projections W_ih x + b_ih + b_hh of nn.LSTM (factory/AutoVC.py:43,77,96;
 * factory/LstmDV.py:12), and the MelGAN WNConv1d / WNConvTranspose1d / ResnetBlock layers
 * (melgan/modules.py:72-130).  BatchNorm and weight norm are folded by the caller.
 *
 * Rows of A outside [0, a_rows_per_utt) read as zero (the convolution's zero padding).
 * Weights are packed [n_pad][k_pad], K contiguous, k_pad = sum_s taps_s * ceil(C_s / KC) * KC with
 * KC = 32 (tf32) or 64 (bf16) channels per k-block, zero filled; n_pad is a multiple of block_n.
 *
 * Poly-phase output (ConvTranspose1d with stride r as a 3-tap convolution, melgan/modules.py:101-112):
 * with out_phases = r the N = r*Cs output columns of GEMM row t are the r consecutive output samples
 * time = r*t + phase, each with Cs channels; all output row indices below are in `time` units and the output
 * index space is B x (r*T).
 */
#define AVC_MAX_SOURCES 4
typedef struct avc_gemm_desc {
  const void* a_ptr[AVC_MAX_SOURCES];   /* activation sources, K-concatenated in order */
  int a_channels[AVC_MAX_SOURCES];      /* C_s */
  long long a_ld[AVC_MAX_SOURCES];      /* elements between consecutive rows (>= C_s, 16-byte multiple) */
  int a_rows_per_utt[AVC_MAX_SOURCES];  /* rows per utterance in the buffer (frames + halo rows) */
  int a_taps[AVC_MAX_SOURCES];          /* taps of source s; 0 = source unused (sources are used in order) */
  int a_tap_t0[AVC_MAX_SOURCES];        /* buffer row that tap 0 reads for output frame 0 (negative => zero pad) */
  int a_tap_dt[AVC_MAX_SOURCES];        /* row step between taps (dilation) */
  const void* w_ptr;         /* packed weights */
  int n_pad, k_pad;
  int dtype;                 /* AVC_DTYPE_TF32, AVC_DTYPE_BF16 or AVC_DTYPE_F16 (operand type of A and W) */
  int B, T;                  /* GEMM row space: B utterances x T frames */
  int N;                     /* real output columns (multiple of 4) */
  const float* bias;         /* [n_pad] fp32 */
  int act;                   /* AVC_ACT_* */
  int out_phases;            /* r >= 1 (0 is read as 1): N = r * Cs, see above */
  void* out;                 /* act(v): [B][out_rows_per_utt][out_ld], written at row out_row0 + time */
  long long out_ld;
  int out_rows_per_utt, out_row0;
  int out_dtype;             /* 0 = fp32, 1 = bf16, 2 = split bf16: hi at column c, lo at column Cs + c (out_ld >= 2Cs), 3 = fp16,
                                4 = split fp16 (two fp16 terms hi | lo, same layout as 2) */
  int out_round_tf32;        /* round fp32 outputs to TF32 (rna) so the next GEMM reads them exactly */
  int out_reflect;           /* also write `out_reflect` reflected halo rows each side (ReflectionPad1d,
                                melgan/modules.py:77,96,121); needs out_row0 >= out_reflect */
  void* out_raw;             /* v before the activation, same dtype as out, rows b*(r*T)+time, ld out_raw_ld (may be NULL) */
  long long out_raw_ld;
  float* out2;               /* act(v) as exact fp32, rows b*(r*T)+time, ld out2_ld (may be NULL) */
  long long out2_ld;
  const float* residual;     /* optional fp32, rows b*(r*T)+time, ld res_ld, added before the activation ... */
  long long res_ld;
  int res_after_act;         /* ... or after it when non-zero (x + relu(bn(conv(..))), factory/MetaPool.py:68,75) */
  int block_n;               /* 64 / 128 / 256; 0 = choose */
  int cta_group;             /* 2 = CTA pairs (tcgen05 cta_group::2, 256-row tiles), 1 = single CTA, 0 = default (2) */
  long long* debug_clk;      /* optional device buffer, 4 x int64 per CTA: clock64 at entry / setup done / accumulator
                                ready / epilogue done, followed by 8 x int64 per tile unit of CTA 0 (first 256 units):
                                producer start / loads issued / MMA thread at unit / accumulator buffer free / first
                                k-block landed / MMAs issued / accumulator ready / epilogue done
                                (profiling aid; NULL in production) */
  int out_raw_dtype;         /* format of out_raw (codes of out_dtype); 0 = same as out_dtype.  The MelGAN "fp16s" layers
                                write LeakyReLU(y) as ONE fp16 value (out, the next k3 convolution's operand) and y itself
                                as two fp16 terms (out_raw, the residual stream, melgan/modules.py:84-85) */
  int out_phase0;            /* this launch produces phases [out_phase0, out_phase0 + out_phase_count) of the out_phases */
  int out_phase_count;       /* poly-phase outputs, N = out_phase_count * Cs (0 = all of them).  A ConvTranspose1d(K = 2r,
                                stride r) needs only two of the three input taps per output phase -- (t-1, t) for phases
                                < r/2, (t, t+1) for the rest -- so it runs as two GEMMs of two taps each instead of one
                                of three with a third of the weights zero (melgan/modules.py:101-112) */
} avc_gemm_desc;

int avc_conv_gemm(const avc_gemm_desc* d, void* stream);

/*
 * Fused MelGAN ResnetBlock (melgan/modules.py:72-85) for the narrow stages, split-bf16 precision (dtype 2):
 *
 *   y = W_sc x + W_1 LeakyReLU( W_3 *_d LeakyReLU(ReflectionPad_d(x)) + b_3 ) + (b_1 + b_sc)
 *
 * One kernel: the dilated k3 convolution, the LeakyReLU between, the k1 convolution and the k1 shortcut; the
 * intermediate stays in shared memory / tensor memory, the block's weights stay resident in shared memory, and each
 * input row is loaded once (the three taps read one shared-memory window through row-shifted descriptors).
 * Same results as the two avc_conv_gemm launches it replaces (up to fp32 summation order).
 *   xa      [B][L + 2*dilation][xa_ld]  LeakyReLU(x) in split bf16 ([hi(C) | lo(C)]), time t at row t + dilation, the
 *           halo rows hold the reflected samples (written by the producer: out / out_row0 / out_reflect below)
 *   x       [B][L][x_ld]                x in split bf16 (the shortcut input)
 *   w       [5][2C][64] bf16: tiles W3 tap 0, 1, 2, W1 (block.4), Wsc (shortcut).  C = 64: tile rows [w_hi (64) ; w_lo (64)]
 *           over the 64 input channels; C = 32: rows [ [w_hi | w_hi] (32) ; [w_lo | 0] (32) ]  (packing.pack_resblock)
 *   bias3   [C] fp32 (block.2);  bias1 [C] fp32 (block.4 bias + shortcut bias)
 *   out     LeakyReLU(y), split bf16 [B][out_rows_per_utt][out_ld] at row out_row0 + t, plus out_reflect mirrored halo
 *           rows each side (the next block's ReflectionPad1d)           -- optional
 *   out_raw y, split bf16 [B][L][out_raw_ld]                            -- optional
 *   out2    LeakyReLU(y), exact fp32 [B*L][out2_ld]                      -- optional, exclusive with out
 * C is 32 or 64, L a multiple of 128, 1 <= dilation <= 16.
 */
typedef struct avc_resblock_desc {
  const void* xa;
  long long xa_ld;
  const void* x;
  long long x_ld;
  const void* w;
  const float* bias3;
  const float* bias1;
  int B, L, C, dilation;
  void* out;
  long long out_ld;
  int out_rows_per_utt, out_row0, out_reflect;
  void* out_raw;
  long long out_raw_ld;
  float* out2;
  long long out2_ld;
} avc_resblock_desc;

int avc_resblock(const avc_resblock_desc* d, void* stream);

/*
 * The same ResnetBlock (melgan/modules.py:72-85) in the "fp16s" precision, reading ONLY the raw residual stream:
 *
 *   y = W_sc x + W_1 LeakyReLU( W_3 *_d LeakyReLU(ReflectionPad_d(x)) + b_3 ) + (b_1 + b_sc)
 *
 * x is stored as two fp16 terms [hi(C) | lo(C)] (AVC out_dtype 4) with its reflected halo rows; the kernel forms the k3
 * operand LeakyReLU(x) itself, in shared memory, as ONE fp16 value per element (two products per weight), keeps the
 * intermediate as two fp16 terms on chip (three products), and reads the shortcut operand from the centre rows of the
 * same window (three products).  HBM traffic per block: one read of x, one write of the output -- half of avc_resblock.
 *   x     [B][L + 2*dilation][x_ld]   time t at row t + dilation; halo rows hold the reflected samples
 *   w     packing.pack_resblock2: tiles W3 tap 0, 1, 2, W1 (block.4), Wsc (shortcut), rows of 64 fp16.
 *         C = 64: every tile [w_hi (64 rows) ; w_lo (64 rows)];  C = 32: W3 tiles rows [w_hi | w_lo] (32 rows),
 *         W1 / Wsc tiles rows [ [w_hi | w_hi] (32) ; [w_lo | 0] (32) ]
 *   bias3 [C] fp32 (block.2);  bias1 [C] fp32 (block.4 bias + shortcut bias)
 *   y     y (y_act = 0) or LeakyReLU(y) (y_act = 1) as two fp16 terms [B][y_rows_per_utt][y_ld] at row y_row0 + t, plus
 *         y_reflect mirrored halo rows each side (the next block's ReflectionPad1d)
 *   out2  LeakyReLU(y), exact fp32 [B*L][out2_ld]           -- exactly one of y / out2 / wav (below)
 * C is 32, 64 or 128, L a multiple of 128, 1 <= dilation <= 16 (C = 128: <= 12).  C = 128 runs on CTA pairs
 * (tcgen05 cta_group::2) with the weights streamed through a TMA ring -- w is then [5][C/64][256][64]: per matrix and
 * 64-channel k-chunk the rows [w_hi[0:64] ; w_lo[0:64] ; w_hi[64:128] ; w_lo[64:128]] -- and writes y only.
 */
typedef struct avc_resblock2_desc {
  const void* x;
  long long x_ld;
  const void* w;
  const float* bias3;
  const float* bias1;
  int B, L, C, dilation;
  void* y;
  long long y_ld;
  int y_rows_per_utt, y_row0, y_reflect, y_act;
  float* out2;
  long long out2_ld;
  long long* debug_clk;      /* optional (C = 128 only): 16 x int64 clock64 stamps per tile of CTA 0, first 64 tiles
                                (profiling aid; NULL in production) */
  /* Fused generator output layer (C = 32; melgan/modules.py:119-124: LeakyReLU, ReflectionPad1d(K/2), Conv1d(C -> 1, K),
   * tanh): with wav != NULL the block's LeakyReLU(y) never leaves the SM -- tiles overlap by K - 1 samples, the K-tap
   * convolution runs on the staged rows in the epilogue, and only wav is written (y and out2 must be NULL). */
  float* wav;                /* [B][L] fp32 */
  const float* mono_w;       /* [K][C] fp32 */
  float mono_bias;
  int mono_taps;             /* K: 3, 5 or 7 */
  /* A padded batch (optional): utterance b has lengths[b] valid rows at this stage, 1 <= lengths[b] <= L.  Only the tiles
   * that hold a valid row run: ceil(lengths[b] / S) of utterance b, S = 128, or 128 - (K - 1) with wav.  tile_start
   * [B + 1] is their prefix table (tile_start[0] = 0, tile_start[b + 1] = tile_start[b] + ceil(lengths[b] / S)) and
   * n_tiles = tile_start[B]; every role of the kernel maps a tile index to its utterance by binary search.  Output rows
   * of skipped tiles are not written.  The last tile of an utterance computes and stores all its rows, rows at and past
   * lengths[b] included (their values are not those of the utterance alone), so the right halo of y for the next
   * block is the caller's: avc_reflect_halo with the same lengths, after this launch.  With wav the output layer
   * reflects at lengths[b] - 1 and writes 0 for the samples of the last tile at and past lengths[b]; wav samples of
   * skipped tiles are not written (zero-fill wav first).  lengths = NULL: every utterance has L rows, as without these
   * fields. */
  const int* lengths;
  const int* tile_start;
  int n_tiles;
} avc_resblock2_desc;

int avc_resblock2(const avc_resblock2_desc* d, void* stream);

/*
 * Recurrence of one uni-directional LSTM layer with hidden size H (multiple of gate_group, >= 64):
 * for t = 0..T-1:  z = xproj[b,t,:] + W_hh h_{t-1}   (xproj = W_ih x_t + b_ih + b_hh, precomputed or fused);  c = s(z_f) c + s(z_i) tanh(z_g);  h = s(z_o) tanh(c)
 * (nn.LSTM semantics, gate order i,f,g,o, zero initial state; factory/AutoVC.py:77,96,103,110;
 * factory/LstmDV.py:12,20).  Each step is a [B x H] x [H x 4H] tensor-core GEMM whose epilogue is the
 * cell update; rows of W_hh and columns of xproj are gate-interleaved in groups of `gate_group`
 * hidden units:  packed index = (u / G) * 4G + gate * G + (u % G).
 */
typedef struct avc_lstm_desc {
  const float* xproj;        /* [B*T][4H] fp32, packed column order, biases included; NULL when xin is given */
  const void* w_hh;          /* [4H][H] packed row order, dtype; dtype 2: [4H][2H] = [w_hi | w_lo] bf16 */
  void* hseq;                /* [B][T][H] dtype (dtype 2: [B][T][2H] split bf16): output sequence and recurrent operand */
  float* hseq_f32;           /* optional exact fp32 copy of the output sequence (may be NULL) */
  float* h_last;             /* optional [B][H] fp32: h_{T-1} only (LstmDV.py:21) (may be NULL) */
  float* c_state;            /* [B][H] fp32 scratch */
  int B, T, H;
  int dtype;
  int gate_group;            /* G: 16 or 32 */
  int persistent;            /* 0 = one launch per step; 1 = one cooperative launch, grid barrier per step */
  unsigned int* grid_barrier;/* 8 KB of scratch (persistent mode): one barrier counter per batch group */
  long long* debug_clk;      /* optional device buffer, 6 (fused input projection: 8) x int64 per (frame, CTA): clock64 stamps (profiling aid) */
  /* Fused input projection (xproj == NULL): z = [x_t | h_{t-1}] [W_ih | W_hh]^T + bias inside the recurrence kernel;
   * the x_t products of frame t+1 run on the tensor pipe while the cell update and grid barrier of frame t are in
   * flight, and the [B*T][4H] fp32 projection is never materialised. */
  const void* xin;           /* [B][T][xin_ld] layer input in the operand format of dtype (dtype 2: [hi | lo] halves) */
  int xin_channels;          /* C_in logical channels (multiple of 8) */
  long long xin_ld;          /* elements per input row */
  const void* w_ih;          /* [4H][Kp] packed row order, Kp = C_in rounded up to the k-block; dtype 2: [4H][2Kp] */
  const float* bias;         /* [4H] fp32 b_ih + b_hh, packed order */
  const int* lengths;        /* optional [B] int32, 1 <= lengths[b] <= T (may be NULL = all T): h_last[b] is h at frame
                                lengths[b] - 1 (a padded batch, pack_padded_sequence semantics), read from hseq_f32, which
                                is then required.  hseq is still written for all T frames; the recurrence is causal, so
                                frames past a length never reach a valid one */
} avc_lstm_desc;

/* Returned by avc_lstm_seq in persistent mode when the grid cannot be co-resident (one wave); nothing was launched. */
#define AVC_ERR_NOT_RESIDENT (-4)

int avc_lstm_seq(const avc_lstm_desc* d, void* stream);

/*
 * Two stacked layers (nn.LSTM(num_layers = 2), factory/AutoVC.py:110) in ONE persistent launch, layer 1 two frames
 * behind layer 0 on the same CTAs: each tick finishes frame t of layer 0 and frame t - 2 of layer 1, and the MMAs of
 * one layer's inputs run while the other layer's cell update and the batch-group barrier are in flight.  Outputs
 * are bit-identical to avc_lstm_seq(l0) followed by avc_lstm_seq(l1).  Requires equal B, T, H, dtype and gate_group,
 * the fused input projection for both layers, l1->xin == l0->hseq, persistent mode, no lengths or h_last; the
 * grid barrier scratch is l0's, and debug_clk (l0's) holds 12 stamps per (tick, CTA) for T + 2 ticks.  Returns
 * AVC_ERR_NOT_RESIDENT, with nothing launched, when the grid cannot be co-resident.
 */
int avc_lstm_seq2(const avc_lstm_desc* l0, const avc_lstm_desc* l1, void* stream);

/*
 * Small-batch form of the same recurrence (B <= 64, split-bf16 or fp16x2 precision): the recurrent weights stay in
 * tensor memory for the whole sequence (4H/128 row blocks x S K-slices, one thread-block cluster per row block
 * reducing its partial sums through distributed shared memory), so a frame moves only h_{t-1}.
 * Same semantics and references as avc_lstm_seq (factory/AutoVC.py:77,96,103,110; factory/LstmDV.py:12,20).
 * Gate rows of w_hh and columns of xproj are packed  p = 128 (u / 32) + 4 (u % 32) + gate.
 * Returns AVC_ERR_NOT_RESIDENT (nothing launched) when the grid cannot be co-resident.
 */
typedef struct avc_lstm_ws_desc {
  const float* xproj;         /* [B*T][4H] fp32, packed column order, biases included */
  const void* w_hh;           /* [4H][2H] = [w_hi | w_lo] bf16, packed row order */
  void* hseq;                 /* [B][T][2H] split bf16: output sequence and recurrent operand */
  float* hseq_f32;            /* optional exact fp32 copy (may be NULL) */
  float* h_last;              /* optional [B][H] fp32: h_{T-1} only (may be NULL) */
  unsigned int* grid_barrier; /* one counter; zeroed by the library */
  int B, T, H;
  long long* debug_clk;       /* optional device buffer, 8 x int64 per (frame, CTA): clock64 stamps (profiling aid) */
  int dtype;                  /* 0 or AVC_DTYPE_BF16X3: as above; AVC_DTYPE_F16 ("fp16x2"): w_hh = [w_hi | w_lo] fp16,
                                 hseq [B][T][H] fp16 */
  const int* lengths;         /* optional [B] int32 (may be NULL): h_last[b] = h at frame lengths[b] - 1, as avc_lstm_desc */
} avc_lstm_ws_desc;

int avc_lstm_seq_ws(const avc_lstm_ws_desc* d, void* stream);

/*
 * A whole STACK of small-batch LSTM layers as one wavefront (B <= 64, fp16 operands): layer l runs two ticks behind layer
 * l - 1, all layers at once on disjoint SMs, so nn.LSTM(num_layers = L) costs T + 2 (L - 1) frame times instead of L x T.
 * Replaces the layer-by-layer loop of factory/LstmDV.py:12,20 (3 x LSTM(80 -> 768), only the last frame of the top
 * layer is used, :21) and factory/Adjust.py:26,40-41.
 *   layer 0:   z_t = xproj0[t]                         + W_hh0 h0_{t-1}      (dense input projection in front, as for
 *                                                                             avc_lstm_seq_ws)
 *   layer l>0: z_t = bias_l + W_ih_l h^{l-1}_t         + W_hh_l h^l_{t-1}    (the W_ih product is issued one tick early,
 *                                                                             off the serial chain of the frame)
 * Every matrix is resident in tensor memory as ONE fp16 term (that is what fits on chip; avc_lstm_seq_ws keeps two).
 * Grid: L x (4H / 128) x 2 CTAs (clusters of 2), all co-resident; H % 128 == 0, H <= 768.  Gate rows of every weight
 * matrix, of xproj0 and of the biases are packed  p = 128 (u / 32) + 4 (u % 32) + gate.
 * Returns AVC_ERR_NOT_RESIDENT (nothing launched) when the grid cannot be co-resident.
 */
#define AVC_STACK_MAX_LAYERS 4
typedef struct avc_lstm_stack_desc {
  const float* xproj0;                        /* [B*T][4H] fp32, packed column order, biases of layer 0 included */
  const void* w_ih[AVC_STACK_MAX_LAYERS];     /* l >= 1: [4H][H] fp16, packed row order (entry 0 unused) */
  const void* w_hh[AVC_STACK_MAX_LAYERS];     /* [4H][H] fp16, packed row order */
  const float* bias[AVC_STACK_MAX_LAYERS];    /* l >= 1: [4H] fp32 = b_ih + b_hh, packed order (entry 0 unused) */
  void* hs;                                   /* scratch [L][T+1][B][H] fp16: frame t+1 of layer l = h^l_t (frame 0 is zeroed
                                                 by the library); on return hs[L-1] holds the top layer's sequence */
  float* h_last;                              /* optional [B][H] fp32: h_{T-1} of the top layer (may be NULL) */
  unsigned int* grid_barrier;                 /* one counter; zeroed by the library */
  int B, T, H, L;
  long long* debug_clk;                       /* optional device buffer, 16 x int64 per (tick, CTA), T + 2 (L - 1) ticks */
  const int* lengths;                         /* optional [B] int32 (may be NULL): h_last[b] = top-layer h at frame
                                                 lengths[b] - 1, as avc_lstm_desc; hs is still written for all T frames */
} avc_lstm_stack_desc;

int avc_lstm_stack_ws(const avc_lstm_stack_desc* d, void* stream);

/*
 * Bidirectional small-H LSTM layer (H <= 64) with the recurrent weights held in shared memory, one warp
 * per (utterance, direction); optionally emits only the down-sampled content code
 * code_j = [h_fwd[jF+F-1] || h_bwd[jF]]  (factory/AutoVC.py:43,54-66).
 *   xproj  [B*T][8H] fp32: columns dir*4H + gate*H + u, biases included
 *   w_hh   [2][4H][H] fp32 (PyTorch row order i,f,g,o)
 *   out    [B][T][2H] (fwd | bwd) in out_dtype (2: [B][T][4H] split bf16), or NULL
 *   codes  [B][T/freq][2H] fp32, or NULL
 *   lengths optional [B] int32 (NULL = every utterance has T frames): utterance b of a padded batch has lengths[b]
 *          valid frames, 1 <= lengths[b] <= T, a multiple of freq when codes are written (the caller checks).  Its
 *          forward direction stops at frame lengths[b] - 1 and its backward direction starts there from the zero state
 *          (nn.utils.rnn.pack_padded_sequence semantics); out rows t >= lengths[b] and codes j >= lengths[b] / freq are
 *          written as 0.  xproj rows past a length are never read.
 */
int avc_bilstm_small(const float* xproj, const float* w_hh, void* out, int out_dtype, int out_round_tf32,
                     float* codes, int B, int T, int H, int freq, void* stream, const int* lengths);

/*
 * out[b,t,:] = [ seq[b, t / div, 0:C1] || vec[b, 0:C2] ]   (channels-last concat with broadcast)
 * Replaces the speaker-code concat of Encoder.forward (factory/AutoVC.py:46-48; div = 1) and the code
 * up-sampling + target-speaker concat of AutoVC.forward (factory/AutoVC.py:197-204; div = freq).
 *   seq [B][T/div][C1] fp32, vec [B][C2] fp32, out [B][T][C1+C2] in out_dtype (2: [B][T][2(C1+C2)] split bf16).
 *   C1, C2 multiples of 4; C2 = 0 (vec NULL) turns it into a pure fp32 -> operand-format conversion.
 */
int avc_concat_bcast(const float* seq, const float* vec, void* out, int B, int T, int C1, int C2, int div,
                     int out_dtype, int out_round_tf32, void* stream);

/*
 * LstmDV tail: e = W h_last + b;  out = e / ||e||_2   (factory/LstmDV.py:21-24).  h [B][K], W [N][K], out [B][N].
 */
int avc_linear_l2norm(const float* h, const float* w, const float* bias, float* out, int B, int K, int N,
                      void* stream);

/*
 * Small fp32 Linear on a handful of rows with both forms of the result: e = W h + b to out_raw and / or e / ||e||_2 to
 * out_normed (either may be NULL).  The classifier twin of the speaker embedder (make_data/factory/LstmDV.py:19-25)
 * needs the un-normalised embedding for its `output` head (`predictions = output(embeds)`, :24) next to the d-vector
 * (`embeds / ||embeds||`, :22-23); the head itself is a second call with out_normed = NULL.
 *   h [B][K], W [N][K], b [N], outputs [B][N]; K multiple of 4, N <= 1024.
 */
int avc_linear_rows(const float* h, const float* w, const float* bias, float* out_raw, float* out_normed, int B, int K,
                    int N, void* stream);

/*
 * Fill the `reflect` halo rows each side of a channels-last buffer [B][rows_per_utt][row_bytes]: row (row0 - k) = row
 * (row0 + k), row (row0 + L - 1 + k) = row (row0 + L - 1 - k), k = 1..reflect -- nn.ReflectionPad1d of the consumer
 * (melgan/modules.py:77,96,121).  avc_conv_gemm can write these rows itself (out_reflect), but only on its general
 * epilogue path; the MelGAN "fp16s" layers keep the GEMM on its branch-free path and add the 2 x reflect rows per
 * utterance with this launch (a few KB).  row_bytes multiple of 16.
 * lengths: optional [B] int32 device (NULL = every utterance has L rows), reflect < lengths[b] <= L: the right halo of
 * utterance b mirrors about row row0 + lengths[b] - 1 instead (a padded batch; its rows row0 + lengths[b] .. are
 * overwritten).  The left halo is the same either way.
 */
int avc_reflect_halo(void* buf, int B, int rows_per_utt, long long row_bytes, int row0, int L, int reflect, void* stream,
                     const int* lengths);

/*
 * Zero the padded tail of every utterance of a channels-last buffer [B][rows_per_utt][row_bytes]: rows
 * row0 + lengths[b] .. row0 + T - 1 of utterance b (lengths: device int32 [B], 1 <= lengths[b] <= T).  A zero is
 * all-zero bits in every operand format (fp32, bf16, fp16, split hi | lo), so after this launch the rows past an
 * utterance's end read as the zero padding the next convolution expects (avc_conv_gemm reads rows outside the buffer
 * as zero, and a padded batch must give each utterance the result of converting it alone).  16-byte stores, nothing
 * else is touched; row_bytes multiple of 16.
 */
int avc_zero_tail(void* buf, int B, int rows_per_utt, long long row_bytes, int row0, int T, const int* lengths,
                  void* stream);

/*
 * in [B][C][L] fp32 (channels-first, the reference's (B, 80, T) mel layout) -> out [B][L + 2*pad][C'] channels-last in
 * out_dtype (C' = C, or 2C for split bf16), with `pad` reflected rows each side (nn.ReflectionPad1d(3) in front of the
 * MelGAN stem, melgan/modules.py:96; `mel.transpose` at conversion.ipynb cell 14).  C multiple of 4, L > pad.
 */
int avc_transpose_pad(const float* in, void* out, int B, int C, int L, int pad, int out_dtype, int out_round_tf32,
                      void* stream);

/*
 * MelGAN output layer: out[b, t] = tanh( bias + sum_k sum_c w[k][c] * x[b, reflect(t + k - K/2), c] )
 * (ReflectionPad1d(3) + WNConv1d(32 -> 1, k7) + Tanh, melgan/modules.py:120-124; the preceding LeakyReLU is applied
 * by the producer).  x [B][L][C] fp32, w [K][C] fp32 (weight norm folded), out [B][L] fp32.  K odd <= 15, C <= 64.
 * lengths: optional [B] int32 device (NULL = all L), K / 2 < lengths[b] <= L: utterance b reflects at its own last
 * sample lengths[b] - 1, and out[b, t] = 0 for t >= lengths[b]; rows of x past lengths[b] are never read.
 */
int avc_conv_to_mono_tanh(const float* x, const float* w, float bias, float* out, int B, int L, int C, int K,
                          void* stream, const int* lengths);

/* ------------------------------------------------------------------------------------------------------------
 * MetaPool / MetaConv glue (factory/MetaPool.py, factory/MetaConv.py, factory/MLPMixer.py).  All inputs are fp32
 * channels-last; `out_dtype` selects the operand format of the output (0 fp32, TF32-rounded when out_round_tf32,
 * 1 bf16, 2 split bf16, 3 fp16 saturating at +-65504).
 * ------------------------------------------------------------------------------------------------------------ */

/* GroupNorm(1, C) statistics (factory/Norm.py:53-60): stats[b] = {mean, 1/sqrt(biased var + eps)} over the n
 * contiguous fp32 elements of sample b. */
int avc_gn_stats(const float* x, float* stats, int B, long long n, float eps, void* stream);

/* MetaPool token mixer + residual (factory/MetaPool.py:7-15,68):
 *   y = x + (AvgPool1d(3,1,1,count_include_pad=False)(GN(x)) - GN(x)) = x + rstd_b * gamma_c * (pool_t(x) - x)
 * x [B][L][C] fp32 -> out_f32 [B][L][C] and/or out_op (operand format). */
int avc_gn_pool_residual(const float* x, const float* stats, const float* gamma, float* out_f32, void* out_op,
                         int out_dtype, int out_round_tf32, int B, int L, int C, void* stream);

/* GroupNorm apply: out = (x - mean_b) * rstd_b * gamma_c + beta_c -> operand format (MetaConv token mixer input,
 * factory/MetaConv.py:66). */
int avc_gn_apply(const float* x, const float* stats, const float* gamma, const float* beta, void* out_op,
                 int out_dtype, int out_round_tf32, int B, int L, int C, void* stream);

/* einops "b c (h p1) (w p2) -> b (h w) (p1 p2 c)" (factory/MLPMixer.py:76-78) of the S x S image whose rows are the
 * CHANNELS and whose columns are the LENGTH axis of a [B][L=S][C=S] channels-last tensor, optionally after
 * GroupNorm(1, S) (stats/gamma/beta may be NULL): tokens [B][(S/p)^2][p*p] in operand format.  S % p == 0, S % 4 == 0
 * and (p*p) % 8 == 0. */
int avc_patchify(const float* a, const float* stats, const float* gamma, const float* beta, void* out_op, int out_dtype,
                 int out_round_tf32, int B, int S, int p, void* stream);

/* Transpose with optional LayerNorm (factory/MLPMixer.py:27-33): x [B][R][C] fp32 -> out_op [B][C][R] (operand
 * format) and/or out_f32 [B][C][R] (the un-normalised values).  ln_axis: 0 none, 1 normalise every ROW over its C
 * entries (gamma/beta indexed by column), 2 normalise every COLUMN over its R entries (gamma/beta indexed by row);
 * biased variance, eps 1e-5.  out_op and out_f32 have R_pad = R rounded up to 8 columns; columns [R, R_pad) are zero.
 * `scratch` holds 2*B*max(R,C) floats; it receives the LayerNorm statistics as (mean, rstd) float pairs, at
 * scratch[2*(b*R + r)] for row r on axis 1 and at scratch[2*(b*C + c)] for column c on axis 2 (unused on axis 0).  They
 * are accumulated as centred sums (Welford, Chan's merge), so their error grows linearly, not quadratically, with
 * |mean| / std. */
int avc_ln_transpose(const float* x, const float* gamma, const float* beta, int ln_axis, void* out_op, int out_dtype,
                     int out_round_tf32, float* out_f32, float* scratch, int B, int R, int C, void* stream);

/* Meta decoder input (factory/MetaPool.py:262-271 feeding Decoder.forward:160-162, which reads the (B, T, 2H+E)
 * tensor as channels = T, length = 2H+E): out[b][f][t] = f < 2H ? codes[b][t / freq][f] : c_trg[b][f - 2H],
 * channels-last [B][2H+E][T] in operand format.  T % 8 == 0 and T % freq == 0. */
int avc_meta_decoder_input(const float* codes, const float* c_trg, void* out_op, int out_dtype, int out_round_tf32,
                           int B, int T, int freq, int H2, int E, void* stream);

/* Content-code down-sampling of the Meta encoders (factory/MetaPool.py:122-133):
 * codes[b][j] = [ out[b][j*freq + freq-1][0:H] || out[b][j*freq][H:2H] ],  out [B][T][2H] fp32. */
int avc_gather_codes(const float* out, float* codes, int B, int T, int H, int freq, void* stream);

/*
 * AdaIN "2" variants (factory/AutoVC2.py, MetaPool2.py, MetaConv2.py).
 * avc_global_stats: stats = {x.mean(), x.std()} over ALL n fp32 elements (torch defaults: Bessel-corrected std), as the
 *   encoder records after each feature_pre_extract layer (factory/AutoVC2.py:57-60).  scratch: 512 doubles.
 * avc_adain: out = (x - x_stats[0]) / x_stats[1] * t_stats[1] + t_stats[0]   (factory/Norm.py:86-94, AutoVC2.py:197-198)
 *   x [rows][C] fp32 -> out_f32 [rows][C] and/or out_op (operand format); the four scalars are read from device memory
 *   so a conversion never synchronises with the host.
 */
int avc_global_stats(const float* x, long long n, float* stats, double* scratch, void* stream);
int avc_adain(const float* x, const float* x_stats, const float* t_stats, float* out_f32, void* out_op, int out_dtype,
              int out_round_tf32, long long rows, int C, void* stream);

/*
 * Per-utterance AdaIN statistics of a padded batch (adain_stats = "utterance"): each utterance is normalised and styled
 * as the reference would do it alone.
 * avc_segment_stats: stats[b] = {mean, Bessel-corrected std} over rows 0 .. lengths[b]-1 (all T rows when lengths is
 *   NULL) x C of x [B][T][C] fp32; lengths device int32 [B], 1 <= lengths[b] <= T; C % 4 == 0, B < 65536.  fp64 partial
 *   sums over chunks of AVC_SEGMENT_CHUNK elements counted from the utterance's first element, added in a fixed order:
 *   the bits of stats[b] depend only on utterance b's valid rows and C (not on B, T, other utterances or the padding,
 *   which is never read).  scratch: 2 * B * ceil(T * C / AVC_SEGMENT_CHUNK) doubles.  Two launches, no host sync.
 * avc_adain_segmented: out[b][t] = (x[b][t] - x_stats[2b]) / x_stats[2b+1] * t_stats[t_stride b + 1]
 *   + t_stats[t_stride b], the operation order of avc_adain; t_stride 0: one style for every utterance, 2: t_stats
 *   [B][2].  With lengths, rows t >= lengths[b] are written as 0 in out_f32 and out_op (the zero padding of the next
 *   k = 5 convolution) and x is not read there.  B = 1, t_stride 0, lengths NULL gives the bits of avc_adain.
 */
#define AVC_SEGMENT_CHUNK 4096
int avc_segment_stats(const float* x, int B, int T, int C, const int* lengths, float* stats, double* scratch,
                      void* stream);
int avc_adain_segmented(const float* x, const float* x_stats, const float* t_stats, int t_stride, const int* lengths,
                        float* out_f32, void* out_op, int out_dtype, int out_round_tf32, int B, int T, int C,
                        void* stream);

/*
 * Batch-statistics BatchNorm: nn.BatchNorm1d in training mode (torch.nn.functional.batch_norm, training=True), which is
 * how the reference's notebooks run every conv + BN layer -- they never call .eval() (conversion.ipynb cells 3 and 8,
 * util/evaluate.py; layers factory/AutoVC.py:26-39,117-171, factory/MetaPool.py:37-43,92-99, factory/Adjust.py:17-20,
 * factory/AutoVC2.py:54-60).  The conv runs unfolded through avc_conv_gemm (its own bias, AVC_ACT_NONE) into
 * v [rows][v_ld] fp32 (out2); these two calls then normalise it.
 *
 * avc_bn_batch_stats: per channel c of v (C channels, C % 4 == 0, rows > 1), over ALL rows:
 *   mean_c, var_c (biased);  scale_shift[0][c] = gamma_c / sqrt(var_c + eps),  scale_shift[1][c] = beta_c - mean_c * scale_c
 *   running_mean_c <- (1 - m) running_mean_c + m mean_c
 *   running_var_c  <- (1 - m) running_var_c  + m var_c * rows / (rows - 1)        (unbiased, as torch)
 *   *num_batches_tracked += 1
 *   m = momentum, or 1 / num_batches_tracked (after the increment) when `cumulative` (nn.BatchNorm1d(momentum=None)).
 *   running_mean / running_var / num_batches_tracked may be NULL (no update; the cumulative average needs all three).
 *   Two launches: fp64 partial sums of v and v^2 per (row chunk, channel) into `scratch`, then one merge per channel in a
 *   fixed order -- the result is bitwise reproducible on a given device.  Every input stays on the device: nothing is
 *   read back to the host.  scratch: 2 + 2 * AVC_BN_MAX_PARTS * C doubles.
 *
 * avc_bn_apply: y = act(scale_c * v + shift_c) with an optional fp32 residual added before the activation or after it
 *   (res_after_act: x + relu(BN(conv)), factory/MetaPool.py:68,75; the postnet's mel + BN(conv), factory/AutoVC.py:206-209).
 *   act: AVC_ACT_NONE / RELU / TANH.  Row r = b * T + t of v, residual and out2; `out` (operand format, the stores of the
 *   GEMM epilogue: out_dtype codes as avc_gemm_desc) at row b * out_rows_per_utt + out_row0 + t.  Any of out / out2.
 */
#define AVC_BN_MAX_PARTS 256
int avc_bn_batch_stats(const float* v, long long rows, int C, long long v_ld, const float* gamma, const float* beta,
                       float eps, float momentum, int cumulative, float* running_mean, float* running_var,
                       long long* num_batches_tracked, float* scale_shift, double* scratch, void* stream);

typedef struct avc_bn_apply_desc {
  const float* v;            /* [B*T][v_ld] fp32 */
  long long v_ld;
  const float* scale_shift;  /* [2][C] fp32 from avc_bn_batch_stats */
  int B, T, C;
  int act;                   /* AVC_ACT_NONE / AVC_ACT_RELU / AVC_ACT_TANH */
  const float* residual;     /* optional fp32 [B*T][res_ld] */
  long long res_ld;
  int res_after_act;         /* add the residual after the activation instead of before it */
  void* out;                 /* optional operand-format output [B][out_rows_per_utt][out_ld] */
  long long out_ld;
  int out_rows_per_utt, out_row0;
  int out_dtype;             /* 0 fp32, 1 bf16, 2 split bf16, 3 fp16, 4 split fp16 */
  int out_round_tf32;
  float* out2;               /* optional exact fp32 [B*T][out2_ld] */
  long long out2_ld;
} avc_bn_apply_desc;

int avc_bn_apply(const avc_bn_apply_desc* d, void* stream);

/*
 * Audio2Mel front end (melgan/modules.py:26-69): reflect-pad by (n_fft - hop)/2, STFT(n_fft, hop, hann, center=False),
 * magnitude, mel filter bank, log10(clamp(., 1e-5)).  The STFT runs as an implicit-GEMM convolution on the tensor cores:
 * the padded signal is viewed as rows of `hop` samples (hop = 256 "channels"), a frame is n_fft / hop = 4 consecutive
 * rows, and the windowed DFT basis is a 4-tap convolution weight with 2 * (n_fft/2 + 1) output channels (avc_conv_gemm);
 * the mel projection is a second avc_conv_gemm with the AVC_ACT_LOG10_CLAMP epilogue.
 *   avc_audio_frames: audio [B][L] fp32 -> out [B][rows][hop] operand format, out row r holds padded samples
 *     [r*hop, (r+1)*hop); padded sample j = audio[reflect(j - pad)], zero past the padded length.
 *   avc_complex_mag: spec [rows][2*bins] fp32 (re | im halves) -> mag [rows][bins_pad] operand format,
 *     sqrt(re^2 + im^2) in the first `bins` channels, zero in the padding channels.
 */
int avc_audio_frames(const float* audio, void* out, int B, long long L, int pad, int hop, int rows, int out_dtype,
                     int out_round_tf32, void* stream);
int avc_complex_mag(const float* spec, void* mag, long long rows, int bins, int bins_pad, int out_dtype,
                    int out_round_tf32, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AVC_B200_H_ */
