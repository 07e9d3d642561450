"""TEST INFRASTRUCTURE — the region members of the store protocol (`regionSum`, `regionCopy`; GpuStore runs them
as one kernel each) for the CPU oracle stores, as plain loops over `getValue` / `setValue`, so that Cube and
ShardedCube (over gloo) run their region queries on machines without a GPU.  The oracle stores themselves are
left as they are; the subclasses below add the two members and keep them through the transforms the tests use
(dice of a Cube, the lowered transforms of a ShardedCube), which build their results with `_as_mine`."""
import itertools

from oracle.store_oracle import OracleStore
from shard_store import OracleShardStore


class _RegionLoops:
    @staticmethod
    def _region_indexes(lens, keep):
        """Cell indices of keep[0] x ... x keep[-1] in product order (keep[d] None = the whole axis)."""
        lists = [range(n) if k is None else [int(i) for i in k] for n, k in zip(lens, keep)]
        for combo in itertools.product(*lists):
            index = 0
            for n, c in zip(lens, combo):
                index = index * n + c
            yield index

    def regionSum(self, lens, keep):
        total = 0
        for index in self._region_indexes(lens, keep):
            total += self.getValue(index)
        return total

    def regionCopy(self, src, lens, keep):
        for index in self._region_indexes(lens, keep):
            self.setValue(index, src.getValue(index))

    def _as_mine(self, other):
        out = type(self)(other.size, other._type, other._defaultValue)
        out._dataMap = other._dataMap
        return out

    def dice(self, oldDimensions, newDimensions):
        return self._as_mine(OracleStore.dice(self, oldDimensions, newDimensions))


class RegionOracleStore(_RegionLoops, OracleStore):
    pass


class RegionOracleShardStore(_RegionLoops, OracleShardStore):
    pass
