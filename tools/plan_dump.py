"""Print the compiled kernel schedules of a model configuration WITHOUT a GPU (plans compile over a CPU arena; nothing is launched):
python tools/plan_dump.py [cfg2|cfg3|cfg4|cfg5] [bf16|fp32] [--train] [--ops] [--fingerprint] [--collect-attn] [--frames T]
                          [--set option=value ...]
Shows launches per entry point, arena sizes, algorithmic FLOPs, and (with --ops) every launch with its dimensions, the stream it
runs on and where the side stream is joined.  `--set` overrides a model option (dropout, num_res_blocks, use_scale_shift_norm...);
a training plan takes its dropout probability from the model.

--fingerprint prints a canonical, pointer-free listing of the compiled plan instead: every launched struct field by field, the
device problem arrays decoded with their ctypes classes, the stream layout, gradient buckets, arena sizes, FLOPs, debug taps and
attention maps.  Each pointer becomes (region, byte offset): an arena, a named parameter, the flat gradient buffer, a packed
weight (its pack problem for training plans, its content hash for host-packed inference weights) or another tensor the plan
keeps (content hash).  Two builds of the compiler that print the same listing launch the same schedule."""
import ast, collections, ctypes as C, hashlib, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "latent-flexible-video-diffusion-modeling_b200"))
import torch as th
from improved_diffusion import _native as N_
from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults

CFG = {"cfg2": (dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1), 1, 5),
       "cfg3": (dict(image_size=128, in_channels=3, num_channels=128, num_res_blocks=1), 1, 4),   # short clip: the CPU arena is real memory
       "cfg4": (dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1), 8, 20),
       "cfg5": (dict(image_size=64, in_channels=4, num_channels=128, num_res_blocks=1), 1, 40)}
argv = sys.argv[1:]
opt = lambda name: argv[argv.index(name) + 1] if name in argv else None
valued = {i + 1 for i, a in enumerate(argv) if a in ("--frames", "--set")}
args = [a for i, a in enumerate(argv) if not a.startswith("--") and i not in valued]
over, B, T = CFG[args[0] if args else "cfg2"]
over = dict(over)
T = int(opt("--frames") or T)
for i, a in enumerate(argv):
    if a == "--set":
        k, v = argv[i + 1].split("=", 1)
        over[k] = ast.literal_eval(v)
prec = args[1] if len(args) > 1 else "bf16"
train, show, fingerprint = "--train" in argv, "--ops" in argv, "--fingerprint" in argv
d = model_and_diffusion_defaults()
d.update(over, diffusion_steps=1000)
d["diffusion_space_kwargs"] = dict(diffusion_space="pixel", pre_encoded=False, pre_encoded_stats_dict=None)
th.manual_seed(0)  # host-packed weights are fingerprinted by content
model, _ = create_model_and_diffusion(**d)
model.precision = prec
S = over["image_size"]
engine = model.engine()

if fingerprint:
    # fdm_rpe_tables_prepare encodes tensor maps through the driver; without a GPU, store the problem array itself in the blob
    def _prepare_stub(problems, count, host_blob, blob_bytes):
        n = count * C.sizeof(N_.RpeTableProblem)
        assert n <= blob_bytes
        C.memmove(C.addressof(host_blob._obj), C.addressof(problems._obj), n)
        return 0
    N_.lib().fdm_rpe_tables_prepare = _prepare_stub

kw = dict(train=True, drop_p=engine.train_dropout()) if train else dict(collect_attn="--collect-attn" in argv)
P = engine._compile(B, T, S, S, th.device("cpu"), **kw)


def fingerprint_lines(P):
    params = dict(model.named_parameters())
    regions = []  # (start, end, label)

    def add(t, label):
        if isinstance(t, th.Tensor) and t.numel():
            regions.append((t.data_ptr(), t.data_ptr() + t.numel() * t.element_size(), label))

    def content(t):
        t = t.detach().contiguous()
        raw = (t.view(th.int16) if t.dtype == th.bfloat16 else t).numpy().tobytes()
        return hashlib.sha1(raw + str((t.dtype, tuple(t.shape))).encode()).hexdigest()[:16]

    add(P.arena, "main"), add(P.stats_arena, "stats"), add(P.bzero_arena, "bzero")
    for name, p in params.items():
        add(p, "param:" + name)
    names = {id(p): n for n, p in params.items()}
    if P.train:
        add(P.pgrad, "pgrad")
        for src, src2, dst, co, ci, k, mode in P.pack_problems:
            add(dst, f"pack:{names[id(src)]}:{names.get(id(src2))}:{mode}")
    if P.drop_philox is not None:
        add(P.drop_philox, "philox")
    for key, t in engine.packed.items():
        add(t, f"hostpack:{key[0]}:{content(t)}")

    def keep_tensors(v):
        if isinstance(v, th.Tensor):
            yield v
        elif isinstance(v, dict):
            for x in v.values():
                yield from keep_tensors(x)
        elif isinstance(v, (list, tuple)):
            for x in v:
                yield from keep_tensors(x)
    arrays = {}  # pointer -> decoded problem array, found through the launches that read them
    problem_cls = {"fdm_grouped_linear": N_.LinearProblem, "fdm_rpe_hidden": N_.RpeHiddenProblem,
                   "fdm_rpe_tables": N_.RpeTableProblem, "fdm_pack_weights": N_.PackProblem,
                   "fdm_rpe_hidden_bwd": N_.RpeHiddenBwdProblem, "fdm_grouped_linear_bwd": N_.LinearBwdProblem}
    for fn, _, ref in P.calls + P.bcalls:
        st = ref._obj
        if fn in problem_cls:
            ptr = st.blob if fn == "fdm_rpe_tables" else st.problems
            arrays[ptr] = (problem_cls[fn] * st.count).from_address(ptr) if st.count else []
    found = {r[0] for r in regions}
    for t in keep_tensors(P.keep):  # other kept tensors (timestep frequencies, ...): by content; problem arrays by their launch
        if t.numel() and t.data_ptr() not in found and t.data_ptr() not in arrays:
            add(t, "keep:" + content(t))
    regions.sort()

    def canon(ptr):
        if not ptr:
            return "null"
        if ptr in arrays:
            return "problems"
        hits = [(s, lab) for s, e, lab in regions if s <= ptr < e]
        if not hits:
            raise AssertionError(f"pointer {ptr:#x} falls in no known region")
        s, lab = max(hits)  # innermost region (a parameter slice of a larger tensor)
        return f"{lab}+{ptr - s}"

    def fields(st):
        out = []
        for name, typ in st._fields_:
            v = getattr(st, name)
            out.append(f"{name}={canon(v) if typ is C.c_void_p else (repr(v) if isinstance(v, float) else v)}")
        return " ".join(out)
    lines = []
    for which, calls in (("fwd", P.calls), ("bwd", P.bcalls if P.train else [])):
        for i, (fn, _, ref) in enumerate(calls):
            st = ref._obj
            lines.append(f"{which} {i} {fn} {fields(st)}")
            if fn in problem_cls:
                ptr = st.blob if fn == "fdm_rpe_tables" else st.problems
                for j, item in enumerate(arrays[ptr]):
                    lines.append(f"    [{j}] {fields(item)}")
    lines.append(f"streams side={P.side_begin}:{P.side_end} join_at={P.join_at} bside={sorted(P.bside)} bjoin_before={P.bjoin_before}")
    if P.train:
        lines.append(f"grad_buckets {P.grad_buckets}")
    lines.append(f"arena main={P.arena_bytes} stats={P.stats_bytes} bzero={P.bzero_bytes}")
    lines.append(f"flops fwd={P.flops} bwd={getattr(P, 'bflops', None)} launches={P.n_launches}")
    for name, (b, Cc, Hh, Ww) in P.taps.items():
        lines.append(f"tap {name} {b.arena}+{b.offset} {Cc}x{Hh}x{Ww}")
    for key, maps in P.attn_maps.items():
        for b, shape in maps:
            lines.append(f"attn_map {key} {b.arena}+{b.offset} {shape}")
    return lines


if fingerprint:
    lines = fingerprint_lines(P)
    print("\n".join(lines))
    print("sha256", hashlib.sha256("\n".join(lines).encode()).hexdigest())
    sys.exit(0)

DIMS = ("N", "B", "T", "HW", "L", "Hin", "Win", "H", "W", "C", "C0", "C1", "Ca", "Cb", "Cw", "Cout", "ksize", "stride", "heads", "count",
        "phases", "upsample", "engine")
print(f"{args[0] if args else 'cfg2'} {prec} B={B} T={T}: params {sum(p.numel() for p in model.parameters()) / 1e6:.2f} M, "
      f"arena {P.arena_bytes / 1e6:.1f} MB, statistics arena {P.stats_bytes / 1e3:.1f} KB")
for title, ops, flops in (("forward", P.ops, P.flops),) + ((("backward", P.bops, P.bflops),) if train else ()):
    cnt = collections.Counter(fn for fn, _, _ in ops)
    print(f"--- {title}: {len(ops)} C-ABI calls, {flops / 1e9:.2f} GFLOP algorithmic")
    print("    " + ", ".join(f"{k} x{v}" for k, v in cnt.most_common()))
    if show:
        for i, (fn, _, f) in enumerate(ops):
            where = "main"
            if title == "forward" and P.side_begin <= i < P.side_end:
                where = "side"
            if title == "backward" and i in P.bside:
                where = "side"
            note = "   <- main stream joins the side stream here" if ((title == "backward" and i == P.bjoin_before) or
                                                                     (title == "forward" and i == P.join_at and P.side_end > P.side_begin)) else ""
            dims = " ".join(f"{k}={f[k]}" for k in DIMS if k in f and not isinstance(f[k], (th.Tensor, tuple)) and f[k] is not None
                            and not hasattr(f[k], "nbytes"))
            print(f"  {i:4d} [{where}] {fn:24s} {dims}{note}")
if train:
    print(f"--- training: {len(P.pack_problems)} weight-pack problems in one launch, parameter-gradient buffer {P.pgrad.numel() * 4 / 1e6:.1f} MB, "
          f"accumulator arena {P.bzero_bytes / 1e3:.1f} KB, side-stream launches {len(P.bside)}, join before op {P.bjoin_before}")
