package muse

/*
#cgo CFLAGS: -I${SRCDIR}/../../../include
#cgo LDFLAGS: -L${SRCDIR}/../.. -lmuse_b200
#include <stdlib.h>
#include "muse_b200.h"
*/
import "C"

import (
	"errors"
	"fmt"
	"os"
	"runtime"
	"sort"
	"strconv"
	"sync"
	"unsafe"
)

var (
	ctxOnce sync.Once
	ctx     *C.muse_ctx
	ctxErr  error
)

func lastError(rc C.int) error {
	return fmt.Errorf("muse_b200: %s (status %d)", C.GoString(C.muse_last_error()), int(rc))
}

// deviceContext creates the process-wide context on device MUSE_DEVICE (default 0; one process per GPU sets it to its
// local rank).
func deviceContext() (*C.muse_ctx, error) {
	ctxOnce.Do(func() {
		dev := 0
		if v := os.Getenv("MUSE_DEVICE"); v != "" {
			d, err := strconv.Atoi(v)
			if err != nil || d < 0 {
				ctxErr = fmt.Errorf("muse_b200: MUSE_DEVICE=%q is not a device index", v)
				return
			}
			dev = d
		}
		if rc := C.muse_ctx_create(C.int(dev), &ctx); rc != C.MUSE_OK {
			ctxErr = lastError(rc)
		}
	})
	return ctx, ctxErr
}

// Group is a collection of uniquely labelled timeseries of one length (go-muse group.go:7-104).
// The values live in a device-resident fp64 slab; label values are dictionary encoded to int32
// ids per key (strings never cross the C boundary).
type Group struct {
	Name     string
	n        int
	registry map[string]int // uid -> index into series
	series   []*Series

	store    *C.muse_group
	gen      uint64                    // bumped whenever the device store is replaced: a Batch bound to an older one rebinds
	cols     []string                  // label key of each device column (the last column is all -1)
	dict     map[string]map[string]int32
	uploaded int

	// sharded groups (exchange.go): index of this block's first series in the whole group, and the label dictionary
	// every process agreed on
	sharded    bool
	shardFirst int64
	fixedDict  map[string][]string
}

// uploadChunk is the number of series handed to muse_group_append per call: the library copies the rows (through its
// pinned staging ring when they sit in pageable Go memory), so nothing larger than one chunk is ever duplicated on the host.
const uploadChunk = 4096

// NewGroup creates a new Group and initializes the timeseries label registry.
func NewGroup(name string) *Group {
	g := &Group{Name: name, registry: make(map[string]int)}
	runtime.SetFinalizer(g, func(g *Group) {
		if g.store != nil {
			C.muse_group_destroy(g.store)
		}
	})
	return g
}

// Length returns the length of all timeseries.
func (g *Group) Length() int { return g.n }

// Add registers time series; errors mirror go-muse group.go:31-56.
func (g *Group) Add(series ...*Series) error {
	for _, s := range series {
		if len(s.lab.Keys()) == 0 {
			return fmt.Errorf("Invalid Series with no labels, %v", s)
		}
		uid := s.UID()
		if _, exists := g.registry[uid]; exists {
			return fmt.Errorf("Series with label:values, %v, already exists within group, %s", uid, g.Name)
		}
		if len(g.registry) == 0 {
			g.n = s.Length()
		} else if s.Length() != g.n {
			return fmt.Errorf("Timeseries has length %d, but current group has length %d", s.Length(), g.n)
		}
		g.registry[uid] = len(g.series)
		g.series = append(g.series, s)
	}
	return nil
}

// FilterByLabelValues returns the series whose values match on every key of labels.
func (g *Group) FilterByLabelValues(labels *Labels) []*Series {
	keys := labels.Keys()
	if len(keys) == 0 {
		return nil
	}
	want := labels.ID(append([]string(nil), keys...))
	var out []*Series
	for _, s := range g.series {
		if s.lab.ID(append([]string(nil), keys...)) == want {
			out = append(out, s)
		}
	}
	return out
}

// syncDevice uploads series added since the last call (muse_group_append copies the rows, so no
// Go pointer is retained by C).
func (g *Group) syncDevice() error {
	c, err := deviceContext()
	if err != nil {
		return err
	}
	keySet := map[string]struct{}{}
	for k := range g.fixedDict { // sharded: every process has the same columns, whatever its own series carry
		keySet[k] = struct{}{}
	}
	for _, s := range g.series {
		for _, k := range s.lab.Keys() {
			keySet[k] = struct{}{}
		}
	}
	keys := make([]string, 0, len(keySet))
	for k := range keySet {
		keys = append(keys, k)
	}
	sort.Strings(keys)
	// a new key needs a column; a key that Remove took from every series keeps its column (all ids -1 now), which groups
	// and filters as an absent key does, so the store is not rebuilt
	known := true
	for _, k := range keys {
		c := sort.SearchStrings(g.cols, k)
		known = known && c < len(g.cols) && g.cols[c] == k
	}
	if g.store == nil || !known {
		if g.store != nil {
			C.muse_group_destroy(g.store)
			g.store = nil
		}
		g.gen++
		g.cols = keys
		g.dict = make(map[string]map[string]int32)
		for _, k := range keys {
			g.dict[k] = make(map[string]int32)
			for i, v := range g.fixedDict[k] {
				g.dict[k][v] = int32(i)
			}
		}
		if rc := C.muse_group_create(c, C.int64_t(g.n), C.int32_t(len(keys)+1), C.int64_t(len(g.series)), &g.store); rc != C.MUSE_OK {
			return lastError(rc)
		}
		if g.shardFirst != 0 {
			if rc := C.muse_group_set_global_offset(g.store, C.int64_t(g.shardFirst)); rc != C.MUSE_OK {
				return lastError(rc)
			}
		}
		g.uploaded = 0
	}
	if g.uploaded == len(g.series) {
		return nil
	}
	nk := len(g.cols) + 1
	rows := make([]float64, 0, uploadChunk*g.n)
	ids := make([]int32, 0, uploadChunk*nk)
	for g.uploaded < len(g.series) {
		end := g.uploaded + uploadChunk
		if end > len(g.series) {
			end = len(g.series)
		}
		rows, ids = rows[:0], ids[:0]
		for _, s := range g.series[g.uploaded:end] {
			rows = append(rows, s.vals...)
			base := len(ids)
			for c := 0; c < nk; c++ {
				ids = append(ids, -1)
			}
			for c, k := range g.cols {
				if v, ok := s.lab.Get(k); ok {
					d := g.dict[k]
					id, seen := d[v]
					if !seen {
						id = int32(len(d))
						d[v] = id
					}
					ids[base+c] = id
				}
			}
		}
		rc := C.muse_group_append(g.store, (*C.double)(unsafe.Pointer(&rows[0])), C.int64_t(end-g.uploaded), C.int64_t(g.n),
			(*C.int32_t)(unsafe.Pointer(&ids[0])))
		if rc != C.MUSE_OK {
			return lastError(rc)
		}
		g.uploaded = end
	}
	return nil
}

// rollChunkBytes bounds the new samples handed to muse_group_roll per call: the library copies them (through its pinned
// staging ring when they sit in pageable Go memory), so nothing larger than one chunk is duplicated on the host.
const rollChunkBytes = 64 << 20

// Roll slides every series forward by k = len(samples[i]) new samples, y <- y[k:] ++ samples[i] for the i-th series in Add
// order: on the device store in place (the store is not sent to the device again) and in each Series' values, which a later
// store rebuild uploads.  Every row holds the same k, 0 <= k <= Length(); the checks come before any device call.  A sharded
// group (SetShard) rolls its own block of series; nothing is exchanged.  When the device fails part-way the store is dropped
// and rebuilt from the unchanged values by the next call that needs it, so a failed Roll has no effect.
func (g *Group) Roll(samples [][]float64) error {
	if len(samples) != len(g.series) {
		return fmt.Errorf("Roll: %d rows of samples for %d series", len(samples), len(g.series))
	}
	if len(samples) == 0 {
		return nil
	}
	k := len(samples[0])
	for i, r := range samples {
		if len(r) != k {
			return fmt.Errorf("Roll: row %d has %d samples, row 0 has %d", i, len(r), k)
		}
	}
	if k > g.n {
		return fmt.Errorf("Roll: %d new samples exceed the series length %d", k, g.n)
	}
	if k == 0 {
		return nil
	}
	if err := g.syncDevice(); err != nil {
		return err
	}
	per := rollChunkBytes / (8 * k)
	if per < 1 {
		per = 1
	}
	if per > len(samples) {
		per = len(samples)
	}
	buf := make([]float64, 0, per*k)
	for first := 0; first < len(samples); first += per {
		end := first + per
		if end > len(samples) {
			end = len(samples)
		}
		buf = buf[:0]
		for _, r := range samples[first:end] {
			buf = append(buf, r...)
		}
		if rc := C.muse_group_roll(g.store, C.int64_t(first), C.int64_t(end-first), (*C.double)(unsafe.Pointer(&buf[0])), C.int64_t(k)); rc != C.MUSE_OK {
			err := lastError(rc)
			C.muse_group_destroy(g.store)
			g.store = nil
			return err
		}
	}
	for i, s := range g.series {
		v := make([]float64, 0, g.n)
		v = append(v, s.vals[k:]...)
		s.vals = append(v, samples[i]...)
	}
	return nil
}

// Remove takes series out of the group, matched by UID (go-muse has no counterpart).  A series that is not a member is an
// error and nothing is removed; a series named twice is removed once.  With a device store the removal is in place
// (muse_group_remove): the remaining series keep their positions, except that the last ones move into the places of
// removed ones, and the Group's series make the same moves (the library's pairs).  Batches stay bound: the store is not
// replaced.  Without a store, or when the device call fails (the store is then dropped and rebuilt by the next call that
// needs it), the remaining series keep their order.  A group that becomes empty forgets its length, as a new Group.
// Remove then Add of the same UID replaces a series; g.Remove(g.FilterByLabelValues(l)...) removes a label set.
// A sharded group (SetShard) cannot remove: ShardScore.Index counts over all shards.
func (g *Group) Remove(series ...*Series) error {
	if g.sharded {
		return errors.New("Remove: a sharded group cannot remove series")
	}
	idx := make(map[int]bool, len(series))
	for _, s := range series {
		i, ok := g.registry[s.UID()]
		if !ok {
			return fmt.Errorf("Series with label:values, %v, is not within group, %s", s.UID(), g.Name)
		}
		idx[i] = true
	}
	if len(idx) == 0 {
		return nil
	}
	if len(idx) == len(g.series) || g.store == nil {
		if g.store != nil {
			C.muse_group_destroy(g.store)
			g.store = nil
		}
		g.removeInOrder(idx)
		return nil
	}
	if err := g.syncDevice(); err != nil {
		return err
	}
	rows := make([]int64, 0, len(idx))
	for i := range idx {
		rows = append(rows, int64(i))
	}
	sort.Slice(rows, func(a, b int) bool { return rows[a] < rows[b] })
	from := make([]int64, len(rows))
	to := make([]int64, len(rows))
	var moved C.int64_t
	if rc := C.muse_group_remove(g.store, (*C.int64_t)(unsafe.Pointer(&rows[0])), C.int64_t(len(rows)), (*C.int64_t)(unsafe.Pointer(&from[0])),
		(*C.int64_t)(unsafe.Pointer(&to[0])), &moved); rc != C.MUSE_OK {
		err := lastError(rc)
		C.muse_group_destroy(g.store)
		g.store = nil
		g.removeInOrder(idx)
		return err
	}
	for _, r := range rows {
		delete(g.registry, g.series[r].UID())
	}
	for j := 0; j < int(moved); j++ {
		g.series[to[j]] = g.series[from[j]]
		g.registry[g.series[to[j]].UID()] = int(to[j])
	}
	m := len(g.series) - len(rows)
	for i := m; i < len(g.series); i++ {
		g.series[i] = nil
	}
	g.series = g.series[:m]
	g.uploaded = m
	return nil
}

// removeInOrder drops the series at the indices in idx from the host lists, keeping the order of the others.
func (g *Group) removeInOrder(idx map[int]bool) {
	kept := g.series[:0]
	for i, s := range g.series {
		if !idx[i] {
			kept = append(kept, s)
		}
	}
	for i := len(kept); i < len(g.series); i++ {
		g.series[i] = nil
	}
	g.series = kept
	g.registry = make(map[string]int, len(kept))
	for i, s := range kept {
		g.registry[s.UID()] = i
	}
	if len(kept) == 0 {
		g.n = 0
	}
}

// keyCols maps label names to device columns; unknown names mean "no series has it", which
// puts every series in one group (labels.go:61-65 skips absent keys).
func (g *Group) keyCols(groupByLabels []string) []int32 {
	if len(groupByLabels) == 0 {
		return nil
	}
	seen := map[string]bool{}
	var cols []int32
	names := append([]string(nil), groupByLabels...)
	sort.Strings(names)
	for _, name := range names {
		if seen[name] {
			continue
		}
		seen[name] = true
		for c, k := range g.cols {
			if k == name {
				cols = append(cols, int32(c))
			}
		}
	}
	if len(cols) == 0 {
		cols = []int32{int32(len(g.cols))}
	}
	return cols
}

// whereCols maps the label set of FilterByLabelValues to device columns and value ids; ok == false when no series can match
// (a key or a value the dictionary does not know).
func (g *Group) whereCols(labels *Labels) (cols, ids []int32, ok bool) {
	for _, k := range labels.Keys() {
		v, _ := labels.Get(k)
		c := sort.SearchStrings(g.cols, k)
		if c == len(g.cols) || g.cols[c] != k {
			return nil, nil, false
		}
		id, seen := g.dict[k][v]
		if !seen {
			return nil, nil, false
		}
		cols = append(cols, int32(c))
		ids = append(ids, id)
	}
	return cols, ids, len(cols) > 0
}

var errNoSeries = errors.New("comparison group is empty")
