"""CPU: where the host code of libp2s_b200.so keeps its state.  Device memory and kernel attributes belong to one CUDA
device, so every launcher takes them from the per-thread, per-device context (`DeviceCtx`, `device_ctx()` in api.cu)
instead of a `static` / `thread_local` of its own: a thread that works on several devices never hands one device's scratch,
error flag or shared-memory limit to another."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'points2surf_b200', 'csrc')

# the only mutable statics: the error message, StageTimer's map, the read-once flags of the three measurement switches
# (P2S_STAGE_TIMING, P2S_TC_WAITSTATS, P2S_VOL_STATS) and the table of device contexts
ALLOWED = sorted([
    ('api.cu', 'thread_local std::string g_last_error'),
    ('api.cu', 'static std::map<std::string, std::pair<double, long>> g_stage'),
    ('api.cu', 'static int e'),
    ('net_tc.cu', 'static int wstats_on'),
    ('volume.cu', 'static int stats'),
    ('api.cu', 'static thread_local std::vector<std::unique_ptr<DeviceCtx>> table'),
])

_TOKENS = re.compile(r'//[^\n]*|/\*.*?\*/|"(?:\\.|[^"\\\n])*"|\'(?:\\.|[^\'\\\n])*\'', re.S)


def _strip(text):
    """C++ source without comments; string and character literals emptied"""
    return _TOKENS.sub(lambda m: ' ' if m.group(0)[0] == '/' else '""', text)


def _mutable_statics(src):
    """declarations that start with `static` or `thread_local` and declare a variable the program can change"""
    out = []
    for m in re.finditer(r'\b(static|thread_local)\b', src):
        if re.search(r'\b(static|thread_local)\s*$', src[:m.start()]):
            continue                                    # second keyword of `static thread_local`
        decl = re.split(r'[;{=]', src[m.start():], maxsplit=1)[0]
        if '(' in decl:
            continue                                    # a function
        decl = ' '.join(re.sub(r'\[[^\]]*\]', '', decl).split())
        words = re.findall(r'[A-Za-z_]\w*|\*|&', decl)
        if 'constexpr' in words or ('const' in words and not {'*', '&'} & set(words[len(words) - words[::-1].index('const'):])):
            continue                                    # const object
        out.append(decl)
    return out


def test_per_device_state_lives_in_the_device_context():
    # the scan itself
    sample = _strip('''
        static int a = 0;                      // mutable
        static thread_local DevBuf t_ws;
        thread_local int* flag = nullptr;
        static const char* roles[6] = {"x"};   // the pointers are mutable
        static const char* const names[2] = {"a", "b"};
        static constexpr int kN = 4;
        static const int kM = 5;
        static void f(int x) { static_assert(true, "s"); }
    ''')
    assert _mutable_statics(sample) == ['static int a', 'static thread_local DevBuf t_ws', 'thread_local int* flag',
                                        'static const char* roles']

    # no .cu file keeps mutable static / thread_local state of its own
    found, attr = [], []
    for path in sorted(glob.glob(os.path.join(CSRC, '*.cu*'))):
        name, src = os.path.basename(path), _strip(open(path).read())
        if name.endswith('.cu'):
            found += [(name, d) for d in _mutable_statics(src)]
        attr += [(name, m.start(), src) for m in re.finditer(r'\bcudaFuncSetAttribute\b', src)]
    assert sorted(found) == ALLOWED, 'mutable static / thread_local state outside the device context: %s' % (
        sorted(set(found) - set(ALLOWED)) or found)
    api = _strip(open(os.path.join(CSRC, 'api.cu')).read())
    assert re.search(r'DeviceCtx& device_ctx\(\) \{\s*static thread_local std::vector<std::unique_ptr<DeviceCtx>> table;', api)

    # shared-memory limits are raised only through DeviceCtx::set_max_dynamic_smem, which remembers them per device
    assert attr
    for name, pos, src in attr:
        assert name == 'api.cu', 'cudaFuncSetAttribute in %s: use DeviceCtx::set_max_dynamic_smem' % name
        start = src.index('void DeviceCtx::set_max_dynamic_smem(')
        assert start < pos < src.index('\n}\n', start), 'cudaFuncSetAttribute outside DeviceCtx::set_max_dynamic_smem'
