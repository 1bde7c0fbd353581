"""Host-side orchestration of the ProGen forward / backward pass over the C-ABI kernels.

Mirrors `ProGenBase.__call__` (reference progen.py:224-233) and its gradient (`jax.value_and_grad`, utils.py:72),
batched over sequences (the reference's `vmap`, utils.py:67).  PyTorch provides device buffers and streams only.

Data layout in HBM (tokens are rows, T = B * seq_len):
  * residual stream: fp32 [T, d], one buffer per LayerNorm input (the residual epilogue of each GEMM writes the next
    one, so nothing is copied and every LN backward still has its input);
  * activations: act dtype (bf16 with mixed_precision, fp32 without), row-major [T, features];
  * q|k|v: one [T, 3*heads*dim_head] buffer, rotated in the QKV GEMM epilogue;
  * parameters, gradients, Adam moments: FLAT fp32 buffers in "engine layout" (ndim > 1 leaves first, then the
    rest; GLU proj_in columns interleaved (value_j, gate_j) so both land in one GEMM tile); a bf16 mirror of the
    parameters feeds the tensor-core GEMMs; SGU spatial weights additionally keep a tril-masked compute copy.
"""
import math
import numpy as np
import torch

from . import lib as L

P = 'pro_gen_base/~/'      # haiku module-path prefix of the reference parameter tree (SURVEY §8(b))
ALIGN = 64                 # every parameter segment starts on a 64-element boundary (TMA needs 16-byte bases)


def layer_kinds(depth, global_mlp_depth, ff_glu):
    """reference progen.py:210-212"""
    out = []
    for i in range(depth):
        use_gmlp = (depth - i) <= global_mlp_depth
        out.append('sgu' if use_gmlp else ('glu' if ff_glu else 'gelu'))
    return out


class ParamSpec:
    __slots__ = ('module', 'name', 'shape', 'decay', 'interleave', 'offset', 'size')

    def __init__(self, module, name, shape, interleave=False):
        self.module, self.name, self.shape = module, name, tuple(shape)
        self.decay = len(shape) > 1                    # optax mask: tree_map(lambda x: x.ndim > 1) — train.py:113
        self.interleave = interleave
        self.size = int(np.prod(shape))
        self.offset = -1


def build_param_specs(cfg):
    d, V, n = cfg['dim'], cfg['num_tokens'], cfg['seq_len']
    inner = cfg['heads'] * cfg['dim_head']
    hid = d * cfg['ff_mult']
    specs = [ParamSpec(P + 'embed', 'embeddings', (V, d))]
    for i, kind in enumerate(layer_kinds(cfg['depth'], cfg['global_mlp_depth'], cfg['ff_glu'])):
        a = P + f'attn{i}/~/'
        specs += [ParamSpec(a + 'layer_norm', 'scale', (d,)),
                  ParamSpec(a + 'linear', 'w', (d, 3 * inner)),
                  ParamSpec(a + 'linear_1', 'w', (inner, d)), ParamSpec(a + 'linear_1', 'b', (d,))]
        f = P + f'ff{i}/~/'
        h_in = hid * 2 if kind == 'glu' else hid
        h_out = hid // 2 if kind == 'sgu' else hid
        glu = kind == 'glu'
        specs += [ParamSpec(f + 'layer_norm', 'scale', (d,)),
                  ParamSpec(f + 'linear', 'w', (d, h_in), interleave=glu), ParamSpec(f + 'linear', 'b', (h_in,), interleave=glu)]
        if kind == 'sgu':
            half = hid // 2
            specs += [ParamSpec(f + 'sgu/~/layer_norm', 'scale', (half,)),
                      ParamSpec(f + 'sgu', 'spatial_weights', (n, n)), ParamSpec(f + 'sgu', 'spatial_biases', (n, 1)),
                      ParamSpec(f + 'sgu/~/linear', 'w', (half, half)), ParamSpec(f + 'sgu/~/linear', 'b', (half,))]
        specs += [ParamSpec(f + 'linear_1', 'w', (h_out, d)), ParamSpec(f + 'linear_1', 'b', (d,))]
    specs += [ParamSpec(P + 'layer_norm', 'scale', (d,)),
              ParamSpec(P + 'linear', 'w', (d, V)), ParamSpec(P + 'linear', 'b', (V,))]
    off = 0
    for s in [s for s in specs if s.decay] + [s for s in specs if not s.decay]:
        s.offset = off
        off += (s.size + ALIGN - 1) // ALIGN * ALIGN
    n_decay = sum((s.size + ALIGN - 1) // ALIGN * ALIGN for s in specs if s.decay)
    return specs, off, n_decay


def _interleave(a):
    """[..., 2H] with columns (value | gate) -> columns (v0, g0, v1, g1, ...)"""
    H = a.shape[-1] // 2
    return np.stack((a[..., :H], a[..., H:]), axis=-1).reshape(a.shape)


def _deinterleave(a):
    return np.concatenate((a[..., 0::2], a[..., 1::2]), axis=-1)


class Engine:
    def __init__(self, cfg, mixed_precision=False, device=None):
        L.require_device()
        self.cfg = cfg
        self.dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self.mp = bool(mixed_precision)
        self.act = torch.bfloat16 if self.mp else torch.float32
        self.act_dt = L.BF16 if self.mp else L.F32
        self.backend = L.BACKEND_TC if self.mp else L.BACKEND_SIMT
        self.kinds = layer_kinds(cfg['depth'], cfg['global_mlp_depth'], cfg['ff_glu'])
        # tensor-core attention kernels: bf16, dim_head 64, 64-aligned windows (checked below — no silent CUDA-core fallback);
        # the fp32 engine (mixed_precision=False) runs the exact CUDA-core kernels
        self.attn_tc = self.mp
        import os
        self.attn_fwd_kind = os.environ.get('PROGEN_ATTN_FWD', 'tcgen05')
        self.attn_bwd_kind = os.environ.get('PROGEN_ATTN_BWD', 'tcgen05')
        if cfg['window_size'] % 128 != 0:
            self.attn_fwd_kind = self.attn_bwd_kind = 'mma'
        d, n, w = cfg['dim'], cfg['seq_len'], cfg['window_size']
        self.d, self.n, self.w, self.V = d, n, w, cfg['num_tokens']
        self.h, self.dh = cfg['heads'], cfg['dim_head']
        self.I = self.h * self.dh
        self.hid = d * cfg['ff_mult']
        if n % w != 0:
            raise L.ProgenError('sequence length must be divisible by the window size')       # progen.py:80
        if self.dh not in (16, 32, 64, 128):
            raise L.ProgenError('dim_head must be one of 16/32/64/128')
        if d % 8 or self.I % 8 or self.V % 8:
            raise L.ProgenError('dim, heads*dim_head and num_tokens must be multiples of 8')
        if self.V > 384:
            raise L.ProgenError('num_tokens > 384 is not supported (embed_bwd keeps num_tokens x 32 fp32 bins in 48 KB of shared memory)')
        if self.mp and self.dh != 64:
            # the tensor-core attention kernels are built for dim_head 64; running another head size on the CUDA-core
            # kernel under mixed_precision would be a silent 10x slowdown, so it is refused (mixed_precision=False runs it)
            raise L.ProgenError(f'mixed_precision needs dim_head == 64 (got {self.dh}); use mixed_precision=False for other head sizes')
        if self.mp and w % 64:
            raise L.ProgenError(f'mixed_precision needs window_size % 64 == 0 (got {w}); use mixed_precision=False')
        if self.mp:
            bad = [k for k, v in dict(dim=d, inner=self.I, seq_len=n, num_tokens=self.V).items() if v % 64]
            if bad:
                raise L.ProgenError(f'mixed_precision (tcgen05 path) needs {bad} to be multiples of 64')
        self.specs, self.n_params_padded, self.n_decay = build_param_specs(cfg)
        self.by_key = {(s.module, s.name): s for s in self.specs}
        self.num_params = sum(s.size for s in self.specs)
        f32 = dict(device=self.dev, dtype=torch.float32)
        self.params = torch.zeros(self.n_params_padded, **f32)
        self.grads = torch.zeros(self.n_params_padded, **f32)
        self.params_lp = torch.zeros(self.n_params_padded, device=self.dev, dtype=torch.bfloat16) if self.mp else None
        self.wm = {}        # layer -> tril-masked compute copy of spatial_weights (act dtype)
        for i, kind in enumerate(self.kinds):
            if kind == 'sgu':
                self.wm[i] = torch.zeros(n, n, device=self.dev, dtype=self.act)
        # rotary tables: fixed_pos_embedding (progen.py:24-28), one (sin, cos) per frequency, computed in float64
        inv_freq = 1.0 / (10000 ** (np.arange(0, self.dh, 2, dtype=np.float64) / self.dh))
        ang = np.arange(n, dtype=np.float64)[:, None] * inv_freq[None, :]
        self.rot_sin = torch.tensor(np.sin(ang), **f32).contiguous()
        self.rot_cos = torch.tensor(np.cos(ang), **f32).contiguous()
        # the same, [dim_head/2, n]: the attention backward reads them one position per thread (coalesced)
        self.rot_sin_t = self.rot_sin.t().contiguous()
        self.rot_cos_t = self.rot_cos.t().contiguous()
        self.B = 0
        self.loss = torch.zeros(1, device=self.dev)       # exists before the first batch: a rank without rows still reports 0
        self.loaded_token = None
        self.on_layer_grads = None        # optional callback(layer_index) fired when a layer's weight gradients are final
        self.lib = L.load()

    def layer_grad_range(self, i):
        """[start, stop) of layer i's ndim>1 parameters inside the flat buffers (contiguous by construction)."""
        pre = (P + f'attn{i}/~/', P + f'ff{i}/~/')
        segs = [s for s in self.specs if s.decay and s.module.startswith(pre)]
        return min(s.offset for s in segs), max(s.offset + (s.size + ALIGN - 1) // ALIGN * ALIGN for s in segs)

    # ------------------------------------------------------------------------------------------ parameters
    def seg(self, buf, module, name):
        s = self.by_key[(module, name)]
        return buf[s.offset:s.offset + s.size]

    def load_params(self, params):
        """haiku-shaped nested dict {module: {name: array}} (numpy or torch) -> flat engine layout on the device."""
        host = np.zeros(self.n_params_padded, np.float32)
        for s in self.specs:
            a = params[s.module][s.name]
            a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
            a = a.astype(np.float32)
            if a.shape != s.shape:
                raise L.ProgenError(f'{s.module}/{s.name}: expected shape {s.shape}, got {a.shape}')
            if s.interleave:
                a = _interleave(a)
            host[s.offset:s.offset + s.size] = a.ravel()
        self.params.copy_(torch.from_numpy(host))
        self.refresh_compute_copies()

    def export_tree(self, buf):
        host = buf.detach().float().cpu().numpy()
        out = {}
        for s in self.specs:
            a = host[s.offset:s.offset + s.size].reshape(s.shape).copy()
            if s.interleave:
                a = _deinterleave(a)
            out.setdefault(s.module, {})[s.name] = a
        return out

    def export_params(self):
        return self.export_tree(self.params)

    def export_grads(self):
        return self.export_tree(self.grads)

    def refresh_compute_copies(self):
        """bf16 mirror of all parameters + tril-masked SGU matrices; call after every parameter change."""
        st = L.stream()
        if self.mp:
            L.check(self.lib.progen_cast_f32(self.params.data_ptr(), self.params_lp.data_ptr(), L.BF16, self.n_params_padded, st),
                    'cast params')
        self.refresh_masked_copies()

    def refresh_masked_copies(self):
        st = L.stream()
        for i, wm in self.wm.items():
            src = self.seg(self.params, P + f'ff{i}/~/sgu', 'spatial_weights')
            L.check(self.lib.progen_tril_cast(src.data_ptr(), wm.data_ptr(), self.act_dt, self.n, st), 'tril_cast')

    def W(self, module, name):
        """GEMM operand view of a parameter: bf16 mirror under mixed precision, fp32 master otherwise."""
        return self.seg(self.params_lp if self.mp else self.params, module, name)

    def Pf(self, module, name):
        return self.seg(self.params, module, name)

    def G(self, module, name):
        return self.seg(self.grads, module, name)

    # ------------------------------------------------------------------------------------------ workspaces
    def ensure_batch(self, B):
        if B == self.B:
            return
        self.B = B
        self.alloc_epoch = getattr(self, 'alloc_epoch', 0) + 1      # activation buffers are re-allocated below: captured
                                                                    # CUDA graphs (Trainer.capture_graph) become invalid
        T = B * self.n
        self.T = T
        d, I, hid = self.d, self.I, self.hid
        dev, act = self.dev, self.act
        A = lambda *shape: torch.empty(*shape, device=dev, dtype=act)
        F = lambda *shape: torch.empty(*shape, device=dev, dtype=torch.float32)
        nl = len(self.kinds)
        self.tok = torch.empty(T, device=dev, dtype=torch.int32)
        self.labels = torch.empty(T, device=dev, dtype=torch.int32)
        self.X = [F(T, d) for _ in range(2 * nl + 1)]           # residual stream at every LN input
        self.lay = []
        for kind in self.kinds:
            s = dict(mean1=F(T), rstd1=F(T), y1=A(T, d), qkv=A(T, 3 * I), att=A(T, I), lse=F(T, self.h),
                     mean2=F(T), rstd2=F(T), y2=A(T, d))
            if kind == 'glu':
                s.update(u=A(T, 2 * hid), hact=A(T, hid))
            else:
                s.update(u=A(T, hid), hact=A(T, hid))
            if kind == 'sgu':
                half = hid // 2
                s.update(mean3=F(T), rstd3=F(T), gn=A(T, half), gp=A(T, half), sg=A(T, half), pj=A(T, half))
            self.lay.append(s)
        self.meanf, self.rstdf, self.yf = F(T), F(T), A(T, d)
        self.logits = F(T, self.V)
        self.dlogits = A(T, self.V)
        self.ce_w = F(T)
        # backward temporaries (shared by all layers)
        self.dres = F(T, d)
        self.dres_lp = A(T, d) if self.mp else self.dres
        self.dy = A(T, d)
        self.dqkv = A(T, 3 * I)
        self.datt = A(T, I)
        self.delta = F(T, self.h)
        self.du = A(T, 2 * hid)
        self.dh_ = A(T, hid)
        half = hid // 2
        if 'sgu' in self.kinds:
            self.dpj, self.dsg, self.dgp, self.dgn = A(T, half), A(T, half), A(T, half), A(T, half)

    # ------------------------------------------------------------------------------------------ GEMM helpers
    def _mm(self, **kw):
        L.gemm(backend=self.backend, in_dtype=self.act_dt, **kw)

    def fwd_gemm(self, x, K, w, N, out, epi=L.EPI_STORE, out_dtype=None, **kw):
        """out[T,N] = x[T,K] @ w[K,N]  (w stored (in, out) like hk.Linear: MN-major B operand)"""
        self._mm(M=self.T, N=N, K=K, A=x, lda=K, B=w, ldb=N, b_mn=True, out=out, ldo=kw.pop('ldo', N), epi=epi,
                 out_dtype=self.act_dt if out_dtype is None else out_dtype, **kw)

    def dgrad_gemm(self, dy, N_out, w, K_in, out, epi=L.EPI_STORE, **kw):
        """out[T,K_in] = dy[T,N_out] @ w[K_in,N_out]^T  (w rows are the output features: K-major B operand)"""
        self._mm(M=self.T, N=K_in, K=N_out, A=dy, lda=N_out, B=w, ldb=N_out, out=out, ldo=kw.pop('ldo', K_in), epi=epi,
                 out_dtype=self.act_dt, **kw)

    def wgrad_gemm(self, x, K_in, dy, N_out, dw):
        """dw[K_in,N_out] += x[T,K_in]^T @ dy[T,N_out]  (both operands MN-major, the token dimension is K)"""
        split = 1
        if self.backend == L.BACKEND_TC:
            bn = 256 if (N_out % 256 == 0) else 128
            tiles = ((K_in + 127) // 128) * ((N_out + bn - 1) // bn)
            split = max(1, min(self.T // 64, 148 // tiles))
        self._mm(M=K_in, N=N_out, K=self.T, A=x, lda=K_in, a_mn=True, B=dy, ldb=N_out, b_mn=True, out=dw, ldo=N_out,
                 epi=L.EPI_ACCUM, out_dtype=L.F32, split_k=split, atomic=split > 1)

    def colsum(self, t, N, out, ld=None):
        L.check(self.lib.progen_colsum(t.data_ptr(), N if ld is None else ld, L.dt(t), out.data_ptr(), self.T, N, L.stream()), 'colsum')

    def ln_fwd(self, x, ldx, scale, y, ldy, mean, rstd, dcols, shift):
        L.check(self.lib.progen_ln_shift_fwd(x.data_ptr(), ldx, L.dt(x), scale.data_ptr(), y.data_ptr(), ldy, L.dt(y),
                                             mean.data_ptr(), rstd.data_ptr(), self.T, dcols, self.n, int(shift), L.stream()), 'ln_fwd')

    # ------------------------------------------------------------------------------------------ forward
    def forward(self, ids):
        """ids: (B, n) integer array/tensor -> self.logits fp32 [T, V]; keeps everything the backward pass needs."""
        B = ids.shape[0]
        self.ensure_batch(B)
        self.tok.copy_(torch.as_tensor(ids).reshape(-1).to(device=self.dev, dtype=torch.int32), non_blocking=True)
        self._forward_device()
        return self.logits

    def _forward_device(self):
        lib, st = self.lib, L.stream()
        cfg, d, I, hid, T, n = self.cfg, self.d, self.I, self.hid, self.T, self.n
        shift = cfg['shift_tokens']
        L.check(lib.progen_embed_fwd(self.tok.data_ptr(), self.Pf(P + 'embed', 'embeddings').data_ptr(), self.X[0].data_ptr(),
                                     T, d, self.V, st), 'embed_fwd')
        for i, kind in enumerate(self.kinds):
            s = self.lay[i]
            a, f = P + f'attn{i}/~/', P + f'ff{i}/~/'
            x0, x1, x2 = self.X[2 * i], self.X[2 * i + 1], self.X[2 * i + 2]
            # ---- LocalAttention (progen.py:73-103)
            self.ln_fwd(x0, d, self.Pf(a + 'layer_norm', 'scale'), s['y1'], d, s['mean1'], s['rstd1'], d, shift)
            self.fwd_gemm(s['y1'], d, self.W(a + 'linear', 'w'), 3 * I, s['qkv'], epi=L.EPI_ROTARY, rot_sin=self.rot_sin,
                          rot_cos=self.rot_cos, seq_len=n, dim_head=self.dh)
            self.attn_fwd(s['qkv'], s['att'], s['lse'])
            self.fwd_gemm(s['att'], I, self.W(a + 'linear_1', 'w'), d, x1, epi=L.EPI_RESIDUAL, bias=self.Pf(a + 'linear_1', 'b'),
                          aux=x0, ldaux=d)
            # ---- FeedForward (progen.py:131-149)
            self.ln_fwd(x1, d, self.Pf(f + 'layer_norm', 'scale'), s['y2'], d, s['mean2'], s['rstd2'], d, shift)
            if kind == 'glu':
                self.fwd_gemm(s['y2'], d, self.W(f + 'linear', 'w'), 2 * hid, s['hact'], epi=L.EPI_GLU, ldo=hid, out2=s['u'],
                              ldo2=2 * hid, bias=self.Pf(f + 'linear', 'b'))
                last, last_k = s['hact'], hid
            else:
                self.fwd_gemm(s['y2'], d, self.W(f + 'linear', 'w'), hid, s['hact'], epi=L.EPI_GELU, out2=s['u'], ldo2=hid,
                              bias=self.Pf(f + 'linear', 'b'))
                last, last_k = s['hact'], hid
            if kind == 'sgu':
                half = hid // 2
                g = f + 'sgu'
                gate = s['hact'][:, half:]
                self.ln_fwd(gate, hid, self.Pf(g + '/~/layer_norm', 'scale'), s['gn'], half, s['mean3'], s['rstd3'], half, False)
                # gate_b = tril(W) @ gn_b for every sequence b; masked K tiles are skipped (causal=1)
                self._mm(M=n, N=half, K=n, A=self.wm[i], lda=n, B=s['gn'], ldb=half, b_mn=True, out=s['gp'], ldo=half,
                         out_dtype=self.act_dt, batch=self.B, b_batch_rows=n, d_batch_rows=n, causal=1)
                L.check(lib.progen_sgu_gate_fwd(s['hact'].data_ptr(), hid, s['gp'].data_ptr(), half,
                                                self.Pf(g, 'spatial_biases').data_ptr(), s['sg'].data_ptr(), half, self.act_dt,
                                                T, half, n, st), 'sgu_gate_fwd')
                self.fwd_gemm(s['sg'], half, self.W(g + '/~/linear', 'w'), half, s['pj'], bias=self.Pf(g + '/~/linear', 'b'))
                last, last_k = s['pj'], half
            self.fwd_gemm(last, last_k, self.W(f + 'linear_1', 'w'), d, x2, epi=L.EPI_RESIDUAL, bias=self.Pf(f + 'linear_1', 'b'),
                          aux=x1, ldaux=d)
        # ---- to_logits (progen.py:219-222)
        xl = self.X[-1]
        self.ln_fwd(xl, d, self.Pf(P + 'layer_norm', 'scale'), self.yf, d, self.meanf, self.rstdf, d, False)
        self.fwd_gemm(self.yf, d, self.W(P + 'linear', 'w'), self.V, self.logits, bias=self.Pf(P + 'linear', 'b'), out_dtype=L.F32)

    def attn_fwd(self, qkv, out, lse):
        if self.attn_tc:
            # two tensor-core forwards: `tcgen05` (default: TMA + tcgen05.mma + TMEM, attn_fwd_ts.cu / attn_tc_pair.cu /
            # attn_tc.cu by window size; needs window % 128 == 0) and `mma` (mma.sync flash kernel, any window % 64 == 0).
            # PROGEN_ATTN_FWD selects.
            if self.attn_fwd_kind == 'tcgen05':
                L.check(self.lib.progen_local_attn_fwd_tc(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), self.B, self.n, self.w,
                                                          self.h, self.dh, L.stream()), 'local_attn_fwd_tc')
                return
            L.check(self.lib.progen_local_attn_fwd(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), self.B, self.n, self.w, self.h,
                                                   self.dh, L.stream()), 'local_attn_fwd')
            return
        L.check(self.lib.progen_local_attn_fwd_simt(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), self.act_dt, self.B, self.n,
                                                    self.w, self.h, self.dh, L.stream()), 'local_attn_fwd')

    def attn_bwd(self, qkv, out, dout, lse, dqkv):
        if self.attn_tc:
            if self.attn_bwd_kind == 'tcgen05':
                L.check(self.lib.progen_local_attn_bwd_tc_ex(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(),
                                                             dqkv.data_ptr(), self.delta.data_ptr(), self.rot_sin.data_ptr(),
                                                             self.rot_cos.data_ptr(), self.rot_sin_t.data_ptr(),
                                                             self.rot_cos_t.data_ptr(), self.B, self.n, self.w, self.h, self.dh, -1,
                                                             L.stream()), 'local_attn_bwd')
                return     # rotary backward is fused into the kernels' epilogues
            L.check(self.lib.progen_local_attn_bwd(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), dqkv.data_ptr(),
                                                   self.delta.data_ptr(), self.rot_sin.data_ptr(), self.rot_cos.data_ptr(), self.B,
                                                   self.n, self.w, self.h, self.dh, L.stream()), 'local_attn_bwd')
            return     # rotary backward is fused into the kernel's epilogue
        L.check(self.lib.progen_local_attn_bwd_simt(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), dqkv.data_ptr(),
                                                    self.delta.data_ptr(), self.act_dt, self.B, self.n, self.w, self.h, self.dh,
                                                    L.stream()), 'local_attn_bwd')

    # ------------------------------------------------------------------------------------------ loss + backward
    def loss_and_grad(self, data, global_batch=None, zero_grads=True):
        """data: (B, n+1) integer rows -> (device scalar loss, grads accumulated into self.grads).
        Mirrors utils.py:61-76: ids = data[:, :-1], labels = data[:, 1:], mean over rows of the masked CE.
        `global_batch` (DDP): scale by 1/global_batch so that a SUM all-reduce yields the global-mean gradient."""
        B = self.load_batch(data)
        self.step_device(global_batch or B, zero_grads)
        return self.loss

    def load_batch(self, data):
        """host (or device) rows (B, n+1) -> self.tok / self.labels; returns B"""
        data = torch.as_tensor(np.asarray(data).astype(np.int32) if not isinstance(data, torch.Tensor) else data)
        B = data.shape[0]
        self.ensure_batch(B)
        dd = data.to(device=self.dev, dtype=torch.int32, non_blocking=True)
        self.tok.copy_(dd[:, :-1].reshape(-1))
        self.labels.copy_(dd[:, 1:].reshape(-1))
        return B

    def step_device(self, global_batch, zero_grads=True):
        """forward + loss + backward on tokens/labels already resident in self.tok / self.labels"""
        self._forward_device()
        lib, st = self.lib, L.stream()
        self.loss.zero_()
        if zero_grads:
            self.grads.zero_()
        L.check(lib.progen_ce_fwd_bwd(self.logits.data_ptr(), L.F32, self.labels.data_ptr(), self.ce_w.data_ptr(),
                                      self.loss.data_ptr(), self.dlogits.data_ptr(), self.act_dt, self.B, self.n, self.V,
                                      1.0 / global_batch, st), 'ce_fwd_bwd')
        self._backward_device()

    def ln_bwd_res(self, dy, x, scale, mean, rstd, dscale, shift, next_bias_grad=None):
        """LN(+shift) backward into the residual-gradient stream; `next_bias_grad` (+= column sums of the updated dres) is
        the bias gradient of the block that is differentiated next (its output bias sees exactly this dres)."""
        L.check(self.lib.progen_ln_shift_bwd(dy.data_ptr(), self.d, self.act_dt, x.data_ptr(), self.d, L.F32, scale.data_ptr(),
                                             mean.data_ptr(), rstd.data_ptr(), self.dres.data_ptr(),
                                             self.dres_lp.data_ptr() if self.mp else 0, self.d, dscale.data_ptr(),
                                             L.ptr(next_bias_grad), self.T, self.d, self.n, int(shift), 1, L.stream()), 'ln_bwd')

    def _backward_device(self):
        lib, st = self.lib, L.stream()
        cfg, d, I, hid, T, n = self.cfg, self.d, self.I, self.hid, self.T, self.n
        shift = cfg['shift_tokens']
        # ---- head
        hw, hl = P + 'linear', P + 'layer_norm'
        self.colsum(self.dlogits, self.V, self.G(hw, 'b'))
        self.wgrad_gemm(self.yf, d, self.dlogits, self.V, self.G(hw, 'w'))
        self.dgrad_gemm(self.dlogits, self.V, self.W(hw, 'w'), d, self.dy)
        self.dres.zero_()
        nl = len(self.kinds)
        self.ln_bwd_res(self.dy, self.X[-1], self.Pf(hl, 'scale'), self.meanf, self.rstdf, self.G(hl, 'scale'), False,
                        next_bias_grad=self.G(P + f'ff{nl - 1}/~/linear_1', 'b'))
        for i in reversed(range(len(self.kinds))):
            kind, s = self.kinds[i], self.lay[i]
            a, f = P + f'attn{i}/~/', P + f'ff{i}/~/'
            x0, x1 = self.X[2 * i], self.X[2 * i + 1]
            dres_lp = self.dres_lp
            # ---- FeedForward backward (d(proj_out bias) = colsum(dres) was produced by the previous LN backward)
            if kind == 'sgu':
                half = hid // 2
                g = f + 'sgu'
                self.wgrad_gemm(s['pj'], half, dres_lp, d, self.G(f + 'linear_1', 'w'))
                self.dgrad_gemm(dres_lp, d, self.W(f + 'linear_1', 'w'), half, self.dpj)
                self.colsum(self.dpj, half, self.G(g + '/~/linear', 'b'))
                self.wgrad_gemm(s['sg'], half, self.dpj, half, self.G(g + '/~/linear', 'w'))
                self.dgrad_gemm(self.dpj, half, self.W(g + '/~/linear', 'w'), half, self.dsg)
                da = self.dh_                                            # gradient wrt gelu output a = [xs | gate], [T, hid]
                L.check(lib.progen_sgu_gate_bwd(self.dsg.data_ptr(), half, s['hact'].data_ptr(), hid, s['gp'].data_ptr(), half,
                                                self.Pf(g, 'spatial_biases').data_ptr(), da.data_ptr(), hid, self.dgp.data_ptr(),
                                                half, self.G(g, 'spatial_biases').data_ptr(), self.act_dt, T, half, n, st),
                        'sgu_gate_bwd')
                # d spatial_weights = tril(sum_b dGp_b @ gn_b^T)
                self._mm(M=n, N=n, K=half, A=self.dgp, lda=half, B=s['gn'], ldb=half, out=self.G(g, 'spatial_weights'), ldo=n,
                         epi=L.EPI_ACCUM, out_dtype=L.F32, batch=self.B, a_batch_rows=n, b_batch_rows=n, batch_reduce=True,
                         atomic=True, tril=True, tril_rows=n)
                # d gn_b = tril(W)^T @ dGp_b
                self._mm(M=n, N=half, K=n, A=self.wm[i], lda=n, a_mn=True, B=self.dgp, ldb=half, b_mn=True, out=self.dgn,
                         ldo=half, out_dtype=self.act_dt, batch=self.B, b_batch_rows=n, d_batch_rows=n, causal=2)
                gate = s['hact'][:, half:]
                L.check(lib.progen_ln_shift_bwd(self.dgn.data_ptr(), half, self.act_dt, gate.data_ptr(), hid, self.act_dt,
                                                self.Pf(g + '/~/layer_norm', 'scale').data_ptr(), s['mean3'].data_ptr(),
                                                s['rstd3'].data_ptr(), 0, da[:, half:].data_ptr(), hid,
                                                self.G(g + '/~/layer_norm', 'scale').data_ptr(), 0, T, half, n, 0, 0, st), 'ln_bwd_sgu')
                L.check(lib.progen_gelu_bwd(da.data_ptr(), s['u'].data_ptr(), self.act_dt, T * hid, st), 'gelu_bwd')
                du, n_in = da, hid
            elif kind == 'glu':
                self.wgrad_gemm(s['hact'], hid, dres_lp, d, self.G(f + 'linear_1', 'w'))
                self.dgrad_gemm(dres_lp, d, self.W(f + 'linear_1', 'w'), hid, self.du, epi=L.EPI_GLU_BWD, ldo=2 * hid,
                                aux=s['u'], ldaux=2 * hid)
                du, n_in = self.du, 2 * hid
            else:
                self.wgrad_gemm(s['hact'], hid, dres_lp, d, self.G(f + 'linear_1', 'w'))
                self.dgrad_gemm(dres_lp, d, self.W(f + 'linear_1', 'w'), hid, self.dh_, epi=L.EPI_GELU_BWD, aux=s['u'], ldaux=hid)
                du, n_in = self.dh_, hid
            self.colsum(du, n_in, self.G(f + 'linear', 'b'))
            self.wgrad_gemm(s['y2'], d, du, n_in, self.G(f + 'linear', 'w'))
            self.dgrad_gemm(du, n_in, self.W(f + 'linear', 'w'), d, self.dy)
            self.ln_bwd_res(self.dy, x1, self.Pf(f + 'layer_norm', 'scale'), s['mean2'], s['rstd2'], self.G(f + 'layer_norm', 'scale'), shift,
                            next_bias_grad=self.G(a + 'linear_1', 'b'))
            # ---- LocalAttention backward
            self.wgrad_gemm(s['att'], I, dres_lp, d, self.G(a + 'linear_1', 'w'))
            self.dgrad_gemm(dres_lp, d, self.W(a + 'linear_1', 'w'), I, self.datt)
            self.attn_bwd(s['qkv'], s['att'], self.datt, s['lse'], self.dqkv)
            if not self.attn_tc:
                L.check(lib.progen_rotary_bwd(self.dqkv.data_ptr(), 3 * I, self.act_dt, self.rot_sin.data_ptr(),
                                              self.rot_cos.data_ptr(), T, 3 * I, n, self.dh, st), 'rotary_bwd')
            self.wgrad_gemm(s['y1'], d, self.dqkv, 3 * I, self.G(a + 'linear', 'w'))
            self.dgrad_gemm(self.dqkv, 3 * I, self.W(a + 'linear', 'w'), d, self.dy)
            self.ln_bwd_res(self.dy, x0, self.Pf(a + 'layer_norm', 'scale'), s['mean1'], s['rstd1'], self.G(a + 'layer_norm', 'scale'), shift,
                            next_bias_grad=self.G(P + f'ff{i - 1}/~/linear_1', 'b') if i > 0 else None)
            if self.on_layer_grads is not None:
                # every weight-matrix gradient of layer i is final: the DDP trainer starts its all-reduce here so the
                # transfer overlaps the backward pass of layers i-1 .. 0
                self.on_layer_grads(i)
        L.check(lib.progen_embed_bwd(self.tok.data_ptr(), self.dres.data_ptr(), self.G(P + 'embed', 'embeddings').data_ptr(),
                                     T, d, self.V, st), 'embed_bwd')
