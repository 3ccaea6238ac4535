"""Device groups without a GPU: the split rule, creation failing loudly, and how the drop-in surface opts in."""
import numpy as np
import pytest

from modal_client_b200 import _backend, _lib, sharding


def split_rule(lengths, nmembers, min_share):
    """The split rule restated: k = min(members, n, max(1, total // min_share)); longest first (stable), dealt over
    0..k-1 in boustrophedon order."""
    lengths = [int(x) for x in lengths]
    n = len(lengths)
    k = min(nmembers, n, max(1, sum(lengths) // min_share)) if n else 0
    owner = [0] * n
    order = sorted(range(n), key=lambda i: -lengths[i])  # sorted() is stable
    for p, i in enumerate(order):
        lap, col = divmod(p, k)
        owner[i] = col if lap % 2 == 0 else k - 1 - col
    return owner, k


def batches():
    rng = np.random.default_rng(7)
    yield "empty", np.zeros(0, np.uint64)
    yield "fewer messages than members", np.array([5 << 20, 1 << 20, 3], np.uint64)
    yield "below the threshold", rng.integers(0, 4096, 500).astype(np.uint64)
    yield "equal lengths", np.full(1000, 4 << 20, np.uint64)
    yield "all empty", np.zeros(64, np.uint64)
    yield "heavy tail", (np.minimum(rng.lognormal(10.4, 2.5, 5000), 1 << 32)).astype(np.uint64)
    yield "one outlier", np.concatenate([np.full(300, 1 << 20, np.uint64), [np.uint64(1 << 33)]])
    for s in range(6):
        yield f"random {s}", rng.integers(0, 64 << 20, int(rng.integers(1, 3000))).astype(np.uint64)


@pytest.mark.parametrize("nmembers", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("min_share", [1, 1 << 20, 256 << 20, 1 << 40])
def test_split_preview_follows_the_rule(nmembers, min_share):
    for name, lengths in batches():
        owner, k = _lib.group_split_preview(lengths, nmembers, min_share)
        want_owner, want_k = split_rule(lengths, nmembers, min_share)
        assert k == want_k, name
        assert owner.tolist() == want_owner, name


def test_default_threshold_is_256_mib_per_member():
    assert _lib.group_split_preview(np.full(8, 32 << 20, np.uint64), 8)[1] == 1  # 256 MiB in all
    assert _lib.group_split_preview(np.full(8, 64 << 20, np.uint64), 8)[1] == 2
    assert _lib.group_split_preview(np.full(64, 64 << 20, np.uint64), 8)[1] == 8


def test_split_preview_deals_as_shard_assignment():
    for name, lengths in batches():
        owner, k = _lib.group_split_preview(lengths, 8, 1)
        if k == 0:
            continue
        plan = sharding.shard_assignment(lengths, k)
        for r in range(k):
            assert np.array_equal(np.flatnonzero(owner == r), plan[r]), (name, r)


def test_split_preview_rejects_bad_arguments():
    with pytest.raises(_lib.B200HashError):
        _lib.group_split_preview([1, 2, 3], 0)


def test_device_group_has_no_cpu_fallback():
    if _lib.load_library().b200h_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    with pytest.raises(_lib.B200HashError, match="b200h_group_create"):
        _lib.DeviceGroup([0, 0])


# ------------------------------------------------------------------------------------------- drop-in surface


@pytest.fixture
def clean_backend(monkeypatch):
    """The backend's module state as a fresh process has it, restored afterwards."""
    for name, value in (("_override", None), ("_devices", None), ("_devices_from_env", False), ("_group", None)):
        monkeypatch.setattr(_backend, name, value)
    for var in ("B200H_DEVICES", "WORLD_SIZE"):
        monkeypatch.delenv(var, raising=False)
    made = []

    class StandInGroup(_lib.DeviceGroup):
        """Records the devices it was asked for; touches no library state."""

        def __init__(self, devices=None, **kw):
            self.devices, self.device, self._g, self._h = devices, 0, None, None
            made.append(self)

    monkeypatch.setattr(_lib, "DeviceGroup", StandInGroup)
    monkeypatch.setattr(_lib, "default_context", lambda device=None: "default context")
    return made


@pytest.mark.parametrize("spec, want", [
    ("all", "all"), ("ALL", "all"), ("0,1,2,3", [0, 1, 2, 3]), (" 0, 0 ", [0, 0]), ([1, 3], [1, 3]), ((0,), [0]),
])
def test_device_specs(clean_backend, spec, want):
    assert _backend._parse_devices(spec) == want


@pytest.mark.parametrize("spec", ["", "gpu0", "0,,1", "0;1", "-1", [], [0, -2], [0.0], [True], "1.5"])
def test_bad_device_specs_are_value_errors(clean_backend, spec):
    with pytest.raises(ValueError):
        _backend.use_devices(spec)


def test_get_context_is_unchanged_when_nothing_is_set(clean_backend):
    assert _backend.get_context() == "default context"
    assert clean_backend == []


def test_use_devices_installs_a_group_and_none_restores_the_default(clean_backend):
    import modal_client_b200

    modal_client_b200.use_devices([0, 1])
    g = _backend.get_context()
    assert isinstance(g, _lib.DeviceGroup) and g.devices == [0, 1]
    assert _backend.get_context() is g  # one group per process
    modal_client_b200.use_devices("all")
    assert _backend.get_context().devices is None  # DeviceGroup(None) = every visible device
    modal_client_b200.use_devices(None)
    assert _backend.get_context() == "default context"


def test_env_var_selects_a_group_on_first_use(clean_backend, monkeypatch):
    monkeypatch.setenv("B200H_DEVICES", "0,1,2,3")
    assert _backend.get_context().devices == [0, 1, 2, 3]
    monkeypatch.setenv("B200H_DEVICES", "4")  # read once
    assert _backend.get_context().devices == [0, 1, 2, 3]


def test_bad_env_var_is_a_value_error(clean_backend, monkeypatch):
    monkeypatch.setenv("B200H_DEVICES", "first")
    with pytest.raises(ValueError):
        _backend.get_context()


def test_groups_are_refused_under_torchrun(clean_backend, monkeypatch):
    monkeypatch.setenv("WORLD_SIZE", "8")
    with pytest.raises(ValueError, match="every rank already owns one GPU"):
        _backend.use_devices("all")
    monkeypatch.setenv("B200H_DEVICES", "all")
    with pytest.raises(ValueError, match="every rank already owns one GPU"):
        _backend.get_context()
    _backend.use_devices(None)  # asking for the default is fine
    assert _backend.get_context() == "default context"


def test_context_pool_returns_the_group(clean_backend):
    _backend.use_devices([0, 0])
    g = _backend.get_context()
    assert _backend.context_pool(3) == [g, g, g]
    assert len(clean_backend) == 1
