"""Pinned byte counts and offsets of every device workspace layout.

The size queries and the view entries only carve: they compute sizes and pointers and touch no memory, so they run
without a GPU, and the views can be handed a fake base address.  A size query that drifts from its carve would let the
kernels write past the end of a caller's workspace; these literals hold every layout to the byte.  The sizes of the
farm's gradient and prediction graphs need a farm, hence a device.
"""
import ctypes

import pytest

NS = (1, 127, 128, 129, 2000, 9000)
EPOCHS = (1, 4, 20)
MODELS = (1, 2, 5, 6, 8)   # SB1, SB2, ST3, FREE1, FREE3
BASE = 1 << 30             # fake 256-aligned workspace address for the view entries
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from psoap_b200 import _build, _lib
    _build.build_library()
    return _lib.load()


def _i64(vals):
    return (ctypes.c_int64 * len(vals))(*vals)


def _i32(vals):
    return (ctypes.c_int32 * len(vals))(*vals)


def _off(p):
    return p.value - BASE


# ---- what each table pins, measured on a library
def lnlike_bytes(lib):
    return [lib.psoap_lnlike_workspace_bytes(N) for N in (0,) + NS]


def schur_bytes(lib):
    return {m: [lib.psoap_schur_workspace_bytes(n, m) for n in NS] for m in (0, 1, 129, 2000)}


def predict_bytes(lib):
    cases = [(1, 0, 300), (2, 0, 129), (3, 0, 1), (1, 1, 300), (2, 1, 2000), (1, 2, None), (3, 2, None)]
    return {(c, mode, m): [lib.psoap_predict_workspace_bytes(c, mode, n, n if m is None else m) for n in NS]
            for c, mode, m in cases}


def lnlike_grad_bytes(lib):
    return {c: [lib.psoap_lnlike_grad_workspace_bytes(c, N) for N in (0,) + NS] for c in (1, 2, 3)}


def chunk_grad_bytes(lib):
    return {(model, ne): [lib.psoap_chunk_lnprob_grad_workspace_bytes(model, N, ne) for N in NS]
            for model in MODELS for ne in EPOCHS}


def chunk_fisher_bytes(lib):
    return {(model, ne): [lib.psoap_chunk_fisher_workspace_bytes(model, N, ne) for N in NS]
            for model in MODELS for ne in EPOCHS}


FARM_NE = (1, 4, 20, 4, 1, 20)


def farm_bytes(lib):
    out = {}
    for nb in (1, 3, 8):
        out[("single", nb)] = lib.psoap_farm_workspace_bytes(len(NS), _i64(NS), _i32(FARM_NE), nb)
        out[("empty", nb)] = lib.psoap_farm_workspace_bytes(1, _i64([0]), _i32([3]), nb)
        for K in (1, 3):
            out[("batched", K, nb)] = lib.psoap_farm_workspace_bytes_batched(len(NS), _i64(NS), _i32(FARM_NE), K, nb)
            for c in (1, 2, 3):
                out[("free", c, K, nb)] = lib.psoap_farm_free_workspace_bytes(c, 20, len(NS), _i64(NS), _i32(FARM_NE),
                                                                               K, nb)
    return out


def lnlike_views(lib):
    out = []
    for N in NS:
        p, T, q, T2 = ctypes.c_void_p(), ctypes.c_int(), ctypes.c_void_p(), ctypes.c_int()
        assert lib.psoap_lnlike_envelope_view(ctypes.c_void_p(BASE), N, ctypes.byref(p), ctypes.byref(T)) == 0
        assert lib.psoap_lnlike_profile_view(ctypes.c_void_p(BASE), N, ctypes.byref(q), ctypes.byref(T2)) == 0
        out.append((_off(p), T.value, _off(q), T2.value))
    return out


def schur_views(lib):
    out = {}
    for m in (0, 129, 2000):
        row = []
        for n in NS:
            r, a, i = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
            assert lib.psoap_schur_views(ctypes.c_void_p(BASE), n, m, ctypes.byref(r), ctypes.byref(a),
                                         ctypes.byref(i)) == 0
            row.append((_off(r), _off(a), _off(i)))
        out[m] = row
    return out


def grad_views(lib):
    out = []
    for N in (0,) + NS:
        k, ld, a = ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_void_p()
        assert lib.psoap_lnlike_grad_views(ctypes.c_void_p(BASE), N, ctypes.byref(k), ctypes.byref(ld),
                                           ctypes.byref(a)) == 0
        out.append((_off(k), ld.value, _off(a)))
    return out


def fisher_views(lib):
    out = {}
    for model in MODELS:
        for ne in (1, 20):
            row = []
            for N in NS:
                fl, kr, Tb = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_int()
                assert lib.psoap_chunk_fisher_views(ctypes.c_void_p(BASE), model, N, ne, ctypes.byref(fl),
                                                    ctypes.byref(kr), ctypes.byref(Tb)) == 0
                row.append((_off(fl), _off(kr), Tb.value))
            out[(model, ne)] = row
    return out


# ---- the pinned values, in the order the functions above measure them (views: offsets from BASE)
LNLIKE =[2399488, 2399488, 2399488, 2399488, 4891904, 67310848, 809949184]
SCHUR = {0: [2268416, 2268416, 2268416, 4367616, 33756416, 149215232],
 1: [4367616, 4367616, 4367616, 6466816, 35855616, 151314688],
 129: [6466816, 6466816, 6466816, 8566016, 37954816, 153413888],
 2000: [35855616, 35855616, 35855616, 37954816, 67344128, 182803712]}
PREDICT = {(1, 0, 300): [10663168, 10663168, 10663168, 13942016, 87371008, 873263360],
 (1, 1, 300): [10663168, 10663168, 10663168, 13942016, 87371008, 873263360],
 (1, 2, None): [4891904, 4891904, 4891904, 10663168, 201561856, 2941202432],
 (2, 0, 129): [10663168, 10663168, 10663168, 13942016, 87371008, 873263360],
 (2, 1, 2000): [73735424, 73735424, 73735424, 80422144, 201561856, 1174887680],
 (3, 0, 1): [4891904, 4891904, 4891904, 7646464, 73735424, 830791936],
 (3, 2, None): [4891904, 4891904, 4891904, 10663168, 201561856, 2941202432]}
LNLIKE_GRAD = {1: [4893696, 4893952, 4894720, 4894720, 10669312, 201842944, 2946478080],
 2: [4894720, 4894976, 4896768, 4896768, 10674432, 202123008, 2951752960],
 3: [4895744, 4896000, 4898816, 4898816, 10679552, 202403584, 2957027840]}
CHUNK_GRAD = {(1, 1): [4894720, 4895488, 4895488, 10670080, 201843712, 2946478848],
 (1, 4): [4895232, 4896000, 4896000, 10670592, 201844224, 2946479360],
 (1, 20): [4898048, 4898816, 4898816, 10673408, 201847040, 2946482176],
 (2, 1): [4895744, 4897536, 4897536, 10675200, 202123776, 2951753728],
 (2, 4): [4896256, 4898048, 4898048, 10675712, 202124288, 2951754240],
 (2, 20): [4899584, 4901376, 4901376, 10679040, 202127616, 2951757568],
 (5, 1): [4897024, 4899840, 4899840, 10680576, 202404608, 2957028864],
 (5, 4): [4897792, 4900608, 4900608, 10681344, 202405376, 2957029632],
 (5, 20): [4903424, 4906240, 4906240, 10686976, 202411008, 2957035264],
 (6, 1): [4894720, 4895488, 4895488, 10670080, 201843712, 2946478848],
 (6, 4): [4894976, 4895744, 4895744, 10670336, 201843968, 2946479104],
 (6, 20): [4904704, 4905472, 4905472, 10680064, 201853696, 2946488832],
 (8, 1): [4896768, 4899584, 4899584, 10680320, 202404352, 2957028608],
 (8, 4): [4897792, 4900608, 4900608, 10681344, 202405376, 2957029632],
 (8, 20): [4925952, 4928768, 4928768, 10709504, 202433536, 2957057792]}
CHUNK_FISHER = {(1, 1): [5944576, 5945344, 5945344, 14866176, 470319104, 8233092864],
 (1, 4): [5945088, 5945856, 5945856, 14866688, 470319616, 8233093376],
 (1, 20): [5947904, 5948672, 5948672, 14869504, 470322432, 8233096192],
 (2, 1): [6339072, 6340864, 6340864, 16444928, 571295232, 10221182976],
 (2, 4): [6339584, 6341376, 6341376, 16445440, 571295744, 10221183488],
 (2, 20): [6342912, 6344704, 6344704, 16448768, 571299072, 10221186816],
 (5, 1): [7389696, 7392512, 7392512, 20647424, 840146432, 15514865408],
 (5, 4): [7390464, 7393280, 7393280, 20648192, 840147200, 15514866176],
 (5, 20): [7396096, 7398912, 7398912, 20653824, 840152832, 15514871808],
 (6, 1): [5288960, 5289728, 5289728, 12243968, 302514432, 4928809728],
 (6, 4): [5682432, 5683200, 5683200, 13817344, 403194368, 6911318528],
 (6, 20): [7791104, 7791872, 7791872, 22221312, 940327424, 17487815424],
 (8, 1): [6077696, 6080512, 6080512, 15400960, 504444160, 8904560640],
 (8, 4): [7259392, 7262208, 7262208, 20123648, 806572032, 14853743616],
 (8, 20): [13595904, 13598720, 13598720, 45367040, 2419432960, 46610715904]}
FARM = {('batched', 1, 1): 809952256,
 ('batched', 1, 3): 2429850624,
 ('batched', 1, 8): 4859698176,
 ('batched', 3, 1): 809957888,
 ('batched', 3, 3): 2429856256,
 ('batched', 3, 8): 6479602176,
 ('empty', 1): 169984,
 ('empty', 3): 169984,
 ('empty', 8): 169984,
 ('free', 1, 1, 1): 809952256,
 ('free', 1, 1, 3): 2429850624,
 ('free', 1, 1, 8): 4859698176,
 ('free', 1, 3, 1): 809957888,
 ('free', 1, 3, 3): 2429856256,
 ('free', 1, 3, 8): 6479602176,
 ('free', 2, 1, 1): 809952512,
 ('free', 2, 1, 3): 2429850880,
 ('free', 2, 1, 8): 4859698432,
 ('free', 2, 3, 1): 809958400,
 ('free', 2, 3, 3): 2429856768,
 ('free', 2, 3, 8): 6479602688,
 ('free', 3, 1, 1): 809952768,
 ('free', 3, 1, 3): 2429851136,
 ('free', 3, 1, 8): 4859698688,
 ('free', 3, 3, 1): 809958912,
 ('free', 3, 3, 3): 2429857280,
 ('free', 3, 3, 8): 6479603200,
 ('single', 1): 809952256,
 ('single', 3): 2429850624,
 ('single', 8): 4859698176}
LNLIKE_VIEWS = [(2398976, 1, 2399232, 1), (2398976, 1, 2399232, 1), (2398976, 1, 2399232, 1), (4891392, 2, 4891648, 2),
 (67310336, 16, 67310592, 16), (809948160, 71, 809948672, 71)]
SCHUR_VIEWS = {0: [(2265088, 2267136, 2267392), (2265088, 2267136, 2267392), (2265088, 2267136, 2267392),
     (4362240, 4366336, 4366592), (33722368, 33755136, 33755392), (149065728, 149211136, 149211392)],
 129: [(6459392, 6465536, 6465792), (6459392, 6465536, 6465792), (6459392, 6465536, 6465792),
       (8556544, 8564736, 8564992), (37916672, 37953536, 37953792), (153260032, 153409536, 153409792)],
 2000: [(35819520, 35854336, 35854592), (35819520, 35854336, 35854592), (35819520, 35854336, 35854592),
        (37916672, 37953536, 37953792), (67276800, 67342336, 67342592), (182620160, 182798336, 182798592)]}
GRAD_VIEWS = [(263168, 256, 4887552), (263168, 256, 4887552), (263168, 256, 4887552), (263168, 256, 4887552),
 (1050624, 512, 10655744), (67125248, 4096, 201510912), (1321540608, 18176, 2940972032)]
FISHER_VIEWS = {(1, 1): [(4894720, 4894976, 1), (4895488, 4895744, 1), (4895488, 4895744, 1), (10670080, 10670336, 2),
          (201843712, 201843968, 16), (2946478848, 2946483968, 71)],
 (1, 20): [(4898048, 4898304, 1), (4898816, 4899072, 1), (4898816, 4899072, 1), (10673408, 10673664, 2),
           (201847040, 201847296, 16), (2946482176, 2946487296, 71)],
 (2, 1): [(4895744, 4896000, 1), (4897536, 4897792, 1), (4897536, 4897792, 1), (10675200, 10675456, 2),
          (202123776, 202124032, 16), (2951753728, 2951758848, 71)],
 (2, 20): [(4899584, 4899840, 1), (4901376, 4901632, 1), (4901376, 4901632, 1), (10679040, 10679296, 2),
           (202127616, 202127872, 16), (2951757568, 2951762688, 71)],
 (5, 1): [(4897024, 4897280, 1), (4899840, 4900096, 1), (4899840, 4900096, 1), (10680576, 10680832, 2),
          (202404608, 202404864, 16), (2957028864, 2957033984, 71)],
 (5, 20): [(4903424, 4903680, 1), (4906240, 4906496, 1), (4906240, 4906496, 1), (10686976, 10687232, 2),
           (202411008, 202411264, 16), (2957035264, 2957040384, 71)],
 (6, 1): [(4894720, 4894976, 1), (4895488, 4895744, 1), (4895488, 4895744, 1), (10670080, 10670336, 2),
          (201843712, 201843968, 16), (2946478848, 2946483968, 71)],
 (6, 20): [(4904704, 4904960, 1), (4905472, 4905728, 1), (4905472, 4905728, 1), (10680064, 10680320, 2),
           (201853696, 201853952, 16), (2946488832, 2946493952, 71)],
 (8, 1): [(4896768, 4897024, 1), (4899584, 4899840, 1), (4899584, 4899840, 1), (10680320, 10680576, 2),
          (202404352, 202404608, 16), (2957028608, 2957033728, 71)],
 (8, 20): [(4925952, 4926208, 1), (4928768, 4929024, 1), (4928768, 4929024, 1), (10709504, 10709760, 2),
           (202433536, 202433792, 16), (2957057792, 2957062912, 71)]}

PINS = [(lnlike_bytes, "LNLIKE"), (schur_bytes, "SCHUR"), (predict_bytes, "PREDICT"),
        (lnlike_grad_bytes, "LNLIKE_GRAD"), (chunk_grad_bytes, "CHUNK_GRAD"), (chunk_fisher_bytes, "CHUNK_FISHER"),
        (farm_bytes, "FARM"), (lnlike_views, "LNLIKE_VIEWS"), (schur_views, "SCHUR_VIEWS"), (grad_views, "GRAD_VIEWS"),
        (fisher_views, "FISHER_VIEWS")]


@pytest.mark.parametrize("measure,name", PINS, ids=[name.lower() for _, name in PINS])
def test_layout_is_pinned(lib, measure, name):
    assert measure(lib) == globals()[name]


# ---- farm graphs: per nbranch, [gradient, prediction (Sigma full, diagonal), draws (1 draw full, 16 draws diagonal)]
FARM_GRAPHS = {
    False: {1: [25401856, 34560512, 29704704, 45242880, 40635136],
            2: [50795264, 64239360, 59383552, 85592064, 81061120],
            4: [101582080, 123597056, 118741248, 166290432, 161913088]},
    True: {1: [25395456, 32120576, 29692672, 42797312, 40531712],
           2: [50787584, 61799424, 59371520, 83146496, 80957696],
           4: [76179712, 91478272, 89050368, 123495680, 121383680]},
}


@gpu
@pytest.mark.parametrize("free", [False, True], ids=["orbit", "free"])
def test_farm_graph_workspace_bytes(lib, free):
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    # N = 120, 140 and 400 (padded 128, 256, 512); the orbit farm holds two proposals of each chunk
    chunks = [synthetic.make_chunk("SB2", ne, npix, seed=s) for ne, npix, s in [(4, 30, 1), (7, 20, 2), (5, 80, 3)]]
    farm = ChunkFarm("SB2", chunks, n_proposals=1 if free else 2, free_velocities=free)
    try:
        f, m = farm._farm, _i64([100, 0, 257])
        got = {nb: [lib.psoap_farm_grad_workspace_bytes(f, nb),
                    lib.psoap_farm_predict_workspace_bytes(f, nb, m, 0),
                    lib.psoap_farm_predict_workspace_bytes(f, nb, m, 1),
                    lib.psoap_farm_predict_draws_workspace_bytes(f, nb, m, 0, 1),
                    lib.psoap_farm_predict_draws_workspace_bytes(f, nb, m, 1, 16)] for nb in (1, 2, 4)}
    finally:
        farm.close()
    assert got == FARM_GRAPHS[free]
