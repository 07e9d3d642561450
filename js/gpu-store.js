// GpuStore — drop-in for src/store/in-memory.js behind the unchanged Cube API.
//
// UNEXECUTED here (no Node.js in the build image, SURVEY.md F4).  Usage in the reference:
//   src/cube.js:12   const InMemoryStore = require('./store/in-memory');
//   becomes          const InMemoryStore = require('olap-gpu-store/js/gpu-store');
// Everything else in cube.js stays as it is: the class below has the members Cube uses
// (constructor, byteLength, size, total, data, getValue, setValue, fill, clone, load,
// reorder, dice, drillUp, drillDown, serialize, deserialize, _type, _defaultValue, _dataMap).  It lowers
// dimension objects to Int32Array maps — exactly the arrays the reference already builds
// (generic.js:243-247, time.js:182-197) — and calls the N-API addon (addon/olap_napi.cc).
const native = require('../addon/build/Release/olap_gpu.node');

const TYPES = { int32: 0, uint32: 1, float32: 2, float64: 3 };
const METHODS = { sum: 0, average: 1, highest: 2, lowest: 3, first: 4, last: 5, product: 6 };
const lens = (dims) => dims.map((d) => d.numItems);

// expr-eval keeps a parsed Expression as a postfix token list already (`expression.tokens`:
// INUMBER / IVAR / IOP1 / IOP2 / IOP3 / IFUNCALL / IEXPR instructions); this rewrites it into the
// text olap_eval() takes (include/olap_gpu.h).  A function call arrives as IVAR(name), the
// arguments, then IFUNCALL(argc); the lazy branches of `a ? b : c` arrive as IEXPR token lists.
function toPostfix(tokens, slots) {
  const stack = [];
  const number = (v) => (Number.isNaN(v) ? '#nan' : v === Infinity ? '#inf' : v === -Infinity ? '#-inf' : `#${v}`);
  for (const t of tokens) {
    if (t.type === 'INUMBER') stack.push({ text: number(t.value) });
    else if (t.type === 'IVAR') stack.push(t.value in slots ? { text: slots[t.value] } : { fn: t.value });
    else if (t.type === 'IEXPR') stack.push({ text: toPostfix(t.value, slots) });
    else if (t.type === 'IOP1') {
      const a = stack.pop();
      stack.push({ text: t.value === '-' ? `${a.text} neg` : t.value === '+' ? a.text : `${a.text} call:${t.value}:1` });
    } else if (t.type === 'IOP2') {
      const b = stack.pop();
      const a = stack.pop();
      stack.push({ text: `${a.text} ${b.text} ${t.value}` });
    } else if (t.type === 'IOP3') {
      const c = stack.pop();
      const b = stack.pop();
      const a = stack.pop();
      stack.push({ text: `${a.text} ${b.text} ${c.text} ?:` });
    } else if (t.type === 'IFUNCALL') {
      const args = stack.splice(stack.length - t.value, t.value);
      const f = stack.pop();
      stack.push({ text: `${args.map((x) => x.text).join(' ')} call:${f.fn}:${t.value}`.trim() });
    } else throw new Error(`Unsupported formula instruction: ${t.type}`);
  }
  return stack.pop().text;
}

class GpuStore {
  constructor(size, type = 'float32', defaultValue = Number.NaN, handle = undefined) {
    if (!Number.isNaN(defaultValue) && defaultValue !== 0)
      throw new Error('Invalid default value, only NaN and 0 are supported');
    if (!(type in TYPES)) throw new Error('Invalid type');
    this._size = size;
    this._type = type;
    this._defaultValue = defaultValue;
    this._h = handle ?? native.create(size, TYPES[type], Number.isNaN(defaultValue) ? 1 : 0, true);
  }

  get size() { return this._size; }
  get byteLength() { return this._size * (this._type === 'float64' ? 8 : 4); }
  get total() { return native.total(this._h); }

  get data() {                       // in-memory.js:30-37: a plain Array of numbers
    const out = new Float64Array(this._size);
    native.download(this._h, out);
    return Array.from(out);
  }
  set data(values) {                 // in-memory.js:39-46 (length check happens natively)
    native.upload(this._h, values instanceof Float32Array ? values : Float64Array.from(values, (v) => v ?? this._defaultValue));
  }
  get dataFloat32() {                // fast path: no Array construction
    const out = new Float32Array(this._size);
    native.download(this._h, out);
    return out;
  }

  get _dataMap() {                   // cube.js:370: Map(index -> value), keys ascending
    const { keys, values } = native.exportSparse(this._h);
    return new Map(Array.from(keys, (k, i) => [Number(k), values[i]]));
  }

  serialize() {                      // in-memory.js:75-101, same record, cells from the device compaction
    const { toBuffer } = require('olap-in-memory/src/serialization');
    const { keys, values } = native.exportSparse(this._h);   // BigInt64Array, Float32Array
    const Typed = { int32: Int32Array, uint32: Uint32Array, float32: Float32Array, float64: Float64Array }[this._type];
    return toBuffer({
      size: this._size,
      type: this._type,
      defaultValue: this._defaultValue,
      indexes: Uint32Array.from(keys, Number),
      dataBuffer: Typed.from(values),
    });
  }
  static deserialize(buffer) {       // in-memory.js:103-116
    const { fromBuffer } = require('olap-in-memory/src/serialization');
    const data = fromBuffer(buffer);
    const store = new GpuStore(data.size, data.type, data.defaultValue);
    native.importSparse(store._h, BigInt64Array.from(data.indexes, BigInt), Float32Array.from(data.dataBuffer));
    return store;
  }

  getValue(index) { return native.getValue(this._h, index); }
  setValue(index, value) { native.setValue(this._h, index, value ?? this._defaultValue); }
  fill(value) { native.fill(this._h, value); }
  clone() { return this._wrap(native.clone(this._h), this._size); }
  _wrap(handle, size) { return new GpuStore(size, this._type, this._defaultValue, handle); }

  drillUp(oldDims, newDims, method = 'sum') {  // in-memory.js:265-334
    if (!(method in METHODS)) throw new Error(`Unsupported aggregation method: ${method}`);
    const maps = newDims.map((nd, i) => Int32Array.from(oldDims[i].getGroupIndexFromRootIndexMap(nd.rootAttribute)));
    const [h] = native.drillUp([this._h], Int32Array.of(METHODS[method]), lens(oldDims), lens(newDims), maps);
    return this._wrap(h, lens(newDims).reduce((m, n) => m * n, 1));
  }

  drillDown(oldDims, newDims, method = 'sum', distributions = null) {  // in-memory.js:336-430
    const maps = oldDims.map((od, i) => Int32Array.from(newDims[i].getGroupIndexFromRootIndexMap(od.rootAttribute)));
    const dist = distributions ? Float64Array.from(distributions, (v) => v ?? Number.NaN) : null;
    const [h] = native.drillDown([this._h], Int32Array.of(METHODS[method] ?? METHODS.last), lens(oldDims), lens(newDims), maps, [dist]);
    return this._wrap(h, lens(newDims).reduce((m, n) => m * n, 1));
  }

  dice(oldDims, newDims) {             // in-memory.js:213-263
    const keep = newDims.map((nd, i) => {
      const oldIdx = oldDims[i].getItemsToIdx();
      return Int32Array.from(nd.getItems(), (item) => oldIdx[item]);
    });
    const [h] = native.dice([this._h], lens(oldDims), lens(newDims), keep);
    return this._wrap(h, lens(newDims).reduce((m, n) => m * n, 1));
  }

  reorder(oldDims, newDims) {          // in-memory.js:178-211
    const newToOld = Int32Array.from(newDims, (nd) => oldDims.indexOf(nd));
    const [h] = native.reorder([this._h], lens(oldDims), newToOld);
    return this._wrap(h, this._size);
  }

  load(other, myDims, hisDims) {       // in-memory.js:139-176
    const maps = hisDims.map((hd, i) => {
      const mine = myDims[i].getItemsToIdx();
      return Int32Array.from(hd.getItems(), (item) => mine[item] ?? -1);
    });
    native.load(this._h, other._h, lens(myDims), lens(hisDims), maps);
  }

  // Region queries: a patched Cube.getTotalForDimensionItems / copyMeasureData lowers the filter to one
  // item-index list per dimension (Int32Array, any order, repeats counted; null = the whole dimension)
  // and makes ONE call instead of a getSingleData / setSingleData per combination (same lowering as store.py).
  regionSum(len, keep) { return native.regionSum(this._h, len, keep); }
  regionCopy(src, len, keep) { native.regionCopy(this._h, src._h, len, keep); }

  // Computed measures (cube.js:331-363): ONE fused kernel instead of a per-cell tree walk.
  // A patched Cube.getData(computedId) calls
  //   GpuStore.evaluate(expression, cellNames, cellNames.map((n) => this.storedMeasures[n]), totals, this.storeSize)
  // in place of the loop at cube.js:353-360 (same arguments the Python host passes, store.py).
  static evaluate(expression, cellNames, stores, totals, size) {
    const totalNames = Object.keys(totals);
    const slots = {};
    cellNames.forEach((n, k) => { slots[n] = `v${k}`; });
    totalNames.forEach((n, k) => { slots[n] = `t${k}`; });
    const out = new Float64Array(size);
    native.evaluate(toPostfix(expression.tokens, slots), stores.map((s) => s._h), Float64Array.from(totalNames, (n) => totals[n]), out);
    return Array.from(out);
  }

  // Computed measures over a region (getTotalForDimensionItems / copyMeasureData of a computed measure): the
  // formula is evaluated only at the region's cells, in the kernel that walks the region (no whole-cube
  // evaluation, nothing per cell on the host).  A formula with an `x__total` variable never gets here.
  static regionEvalSum(expression, cellNames, stores, len, keep) {
    return native.regionEvalSum(cellProgram(expression, cellNames), stores.map((s) => s._h), len, keep);
  }
  static regionEvalCopy(target, expression, cellNames, stores, len, keep) {
    native.regionEvalCopy(target._h, cellProgram(expression, cellNames), stores.map((s) => s._h), len, keep);
  }

  // getStatus / getStatusMap of a computed measure (cube.js:368-389): one kernel each.
  static statusMerge(stores, size) {
    const out = new Uint8Array(size);
    native.statusMerge(stores.map((s) => s._h), out);
    return Array.from(out);
  }
  static statusMap(stores) {
    const { keys, values, isInt } = native.statusMap(stores.map((s) => s._h));
    const out = new Map();
    keys.forEach((k, j) => out.set(Number(k), isInt[j] ? values[j] | 0 : values[j]));
    return out;
  }

  // Batched forms used by a patched Cube to serve all measures with one launch.
  static drillUpMany(stores, oldDims, newDims, methods) {
    const maps = newDims.map((nd, i) => Int32Array.from(oldDims[i].getGroupIndexFromRootIndexMap(nd.rootAttribute)));
    const size = lens(newDims).reduce((m, n) => m * n, 1);
    return native
      .drillUp(stores.map((s) => s._h), Int32Array.from(methods, (m) => METHODS[m ?? 'sum']), lens(oldDims), lens(newDims), maps)
      .map((h, i) => stores[i]._wrap(h, size));
  }
}

function cellProgram(expression, cellNames) {
  const slots = {};
  cellNames.forEach((n, k) => { slots[n] = `v${k}`; });
  return toPostfix(expression.tokens, slots);
}

module.exports = GpuStore;
